// K4 — top-k proposal selection: radix select + ordered compaction + stable LSD sort.
//
// Replaces /root/reference/filter.py:160-161 (full CPU sort of all N candidate scores) for the
// only part rank.py ever reads, the first k rows (/root/reference/rank.py:294).
//
// Order contract (SURVEY §8 a11): score descending, ties by position ascending — exactly
// torch.sort(descending=True, stable=True).  Achieved without a 64-bit composite key:
//   1. map score -> uint32 key, ascending key == descending score (-0.0 folded into +0.0);
//   2. three histogram passes (11+11+10 bits) find T = the k-th smallest key and
//      less = #{key < T}; r = k - less elements equal to T are still needed;
//   3. an ORDERED compaction (per-tile counts -> scan -> write) emits, in position order, every
//      element with key < T and the first r elements with key == T;
//   4. a STABLE 4x8-bit LSD radix sort by key alone keeps equal keys in position order.
// All kernels are HBM streaming passes over `score` (5 reads of 4*M bytes) or over the k
// survivors; the algorithmic figure is a single 4*M read + 12*k out (SURVEY §8d).
//
// Running top-k over owner slabs (eps_topk_select2_f32): the scores are the VIRTUAL concatenation of
// two segments — A = the running list (position order), B = the new slab — and steps 1-3 are run
// without step 4: the survivors come out in position order, which is all the next slab needs (the tie
// rule only looks at positions).  One stable sort at the very end (eps_topk_f32 with k == M) orders
// the final list, instead of two sorts and two selections per slab.
#include "eps_common.cuh"

namespace eps {

constexpr int TK_THREADS = 256;
constexpr int TK_TILE = 4096;      // elements per block in count / write kernels
constexpr int SORT_TILE = 2048;    // elements per block in the LSD sort

struct TopkState {
  uint32_t prefix;      // bits of T found so far
  uint32_t k_rem;       // rank still to resolve inside the current bucket (1-based)
  uint32_t less_total;  // #{key < prefix-bucket}
  uint32_t need_eq;     // r, written after the last pass
};

// scores = segment A (na elements) followed by segment B; position i of the concatenation
struct ScoreSrc {
  const float *a;
  long long na;
  const float *b;
  __device__ __forceinline__ float at(long long i) const {
    return i < na ? __ldg(a + i) : __ldg(b + (i - na));
  }
  // elements i .. i+3 (those < M; the rest 0): one 128-bit load when the four lie in one segment and
  // the address is 16-byte aligned, scalar loads otherwise (segment boundary, ragged end, odd offsets)
  __device__ __forceinline__ void load4(long long i, long long M, float out[4]) const {
    if (i + 3 < M && (i + 3 < na || i >= na)) {
      const float *p = i >= na ? b + (i - na) : a + i;
      if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(p));
        out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
        return;
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) out[q] = i + q < M ? at(i + q) : 0.f;
  }
};

__device__ __forceinline__ uint32_t score_key(float s) {
  uint32_t b = __float_as_uint(s + 0.0f);               // -0.0 -> +0.0
  uint32_t asc = b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);  // ascending float order
  return ~asc;                                          // ascending key == descending score
}

template <int PASS>
__device__ __forceinline__ bool pass_match(uint32_t key, uint32_t prefix) {
  if (PASS == 0) return true;
  if (PASS == 1) return (key >> 21) == (prefix >> 21);
  return (key >> 10) == (prefix >> 10);
}
template <int PASS>
__device__ __forceinline__ uint32_t pass_digit(uint32_t key) {
  if (PASS == 0) return key >> 21;
  if (PASS == 1) return (key >> 10) & 0x7ffu;
  return key & 0x3ffu;
}

// Lanes whose element cannot be the k-th (outside the prefix bucket of the earlier passes, or — pass 0 of a
// running select — worse than the previous k-th key `prune_key`) do not take part.  MATCH.ANY is the
// expensive instruction here (it paces the kernel at ~2 TB/s when issued per element), so it is only used
// when many lanes take part (tie-heavy CN scores would serialise plain shared atomics); a warp with no
// participant skips everything, one with a few issues plain atomics.
template <int PASS>
__global__ void __launch_bounds__(TK_THREADS)
topk_hist_kernel(const ScoreSrc score, long long M, const TopkState *state,
                 const uint32_t *__restrict__ prune_key, uint32_t *__restrict__ hist /*[2048]*/) {
  __shared__ uint32_t sh[2048];
  for (int i = threadIdx.x; i < 2048; i += TK_THREADS) sh[i] = 0;
  __syncthreads();
  const uint32_t prefix = PASS ? state->prefix : 0;
  const uint32_t prune = (PASS == 0 && prune_key) ? *prune_key : 0xffffffffu;
  const int lane = lane_id();
  const long long stride = (long long)gridDim.x * TK_THREADS * 4;
  // whole warps iterate together (warp-uniform trip count); two 128-bit loads in flight per lane
  const long long start = ((long long)blockIdx.x * TK_THREADS + threadIdx.x) * 4;
  for (long long i = start; i - lane * 4 < M; i += 2 * stride) {
    float sc[2][4];
    score.load4(i, M, sc[0]);
    score.load4(i + stride, M, sc[1]);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const long long j0 = i + h * stride;
      if (j0 - lane * 4 >= M) break;                         // warp-uniform
      uint32_t keys[4];
      bool oks[4], any_ok = false;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        keys[q] = score_key(sc[h][q]);
        oks[q] = j0 + q < M && pass_match<PASS>(keys[q], prefix) && keys[q] <= prune;
        any_ok |= oks[q];
      }
      if (__ballot_sync(FULL, any_ok) == 0) continue;          // nobody in these 128 elements takes part
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint32_t key = keys[q];
        const bool ok = oks[q];
        const unsigned part = __ballot_sync(FULL, ok);
        if (part == 0) continue;
        const uint32_t d = ok ? pass_digit<PASS>(key) : 0x10000u;
        if (__popc(part) <= 8) {
          if (ok) atomicAdd(&sh[d], 1u);
        } else {
          const unsigned peers = __match_any_sync(FULL, d);
          if (ok && lane == (__ffs(peers) - 1)) atomicAdd(&sh[d], (uint32_t)__popc(peers));
        }
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2048; i += TK_THREADS)
    if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

// one block of 256 threads: thread t owns bins [8t, 8t+8); block scan of the per-thread totals, then
// the single thread whose range contains the k_rem-th element walks its eight bins
template <int PASS>
__global__ void __launch_bounds__(256) topk_pick_kernel(TopkState *state, const uint32_t *hist, uint32_t k,
                                                        uint32_t *kth_key_out) {
  constexpr int NB = (PASS == 2) ? 1024 : 2048;
  constexpr int PER = NB / 256;
  constexpr int SHIFT = (PASS == 0) ? 21 : (PASS == 1 ? 10 : 0);
  __shared__ uint32_t wtot[8];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const uint32_t k_rem = (PASS == 0) ? k : state->k_rem;
  const uint32_t less = (PASS == 0) ? 0 : state->less_total;
  const uint32_t prefix = (PASS == 0) ? 0 : state->prefix;
  uint32_t c[PER], mine = 0;
#pragma unroll
  for (int q = 0; q < PER; ++q) { c[q] = hist[t * PER + q]; mine += c[q]; }
  uint32_t inc = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(FULL, inc, d);
    if (lane >= d) inc += y;
  }
  if (lane == 31) wtot[warp] = inc;
  __syncthreads();
  uint32_t base = 0;
  for (int w = 0; w < warp; ++w) base += wtot[w];
  const uint32_t before = base + inc - mine;       // elements in bins below this thread's range
  // the k_rem-th element (1-based) lies in the first bin d with cum(<=d) >= k_rem
  if (before < k_rem && k_rem <= before + mine) {
    uint32_t cum = before;
    int q = 0;
    for (; q < PER - 1; ++q) {
      if (cum + c[q] >= k_rem) break;
      cum += c[q];
    }
    const uint32_t d = (uint32_t)(t * PER + q);
    state->prefix = prefix | (d << SHIFT);
    state->k_rem = k_rem - cum;
    state->less_total = less + cum;
    if (PASS == 2) {
      state->need_eq = k_rem - cum;
      if (kth_key_out) *kth_key_out = prefix | (d << SHIFT);      // the k-th key: prune bound of the next select
    }
  }
}

__global__ void __launch_bounds__(TK_THREADS)
topk_count_kernel(const ScoreSrc score, long long M, const TopkState *state,
                  uint32_t *__restrict__ blk_less, uint32_t *__restrict__ blk_eq) {
  const uint32_t T = state->prefix;
  const long long base = (long long)blockIdx.x * TK_TILE;
  uint32_t nl = 0, ne = 0;
#pragma unroll
  for (int t = 0; t < TK_TILE; t += TK_THREADS * 4) {
    const long long i = base + t + threadIdx.x * 4;
    float v[4];
    score.load4(i, M, v);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (i + q < M) {
        const uint32_t key = score_key(v[q]);
        nl += key < T;
        ne += key == T;
      }
    }
  }
  __shared__ uint32_t sl[TK_THREADS / 32], se[TK_THREADS / 32];
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    nl += __shfl_xor_sync(FULL, nl, o);
    ne += __shfl_xor_sync(FULL, ne, o);
  }
  if (lane_id() == 0) { sl[threadIdx.x >> 5] = nl; se[threadIdx.x >> 5] = ne; }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t a = 0, b = 0;
    for (int w = 0; w < TK_THREADS / 32; ++w) { a += sl[w]; b += se[w]; }
    blk_less[blockIdx.x] = a;
    blk_eq[blockIdx.x] = b;
  }
}

// single-block exclusive scan of `a` (and optionally `b`) in place
__global__ void __launch_bounds__(1024)
scan_exclusive_kernel(uint32_t *a, uint32_t *b, long long n) {
  __shared__ uint32_t sa[1024], sb[1024];
  const int t = threadIdx.x;
  const long long per = (n + 1023) / 1024;
  const long long lo = min(n, (long long)t * per), hi = min(n, lo + per);
  uint32_t xa = 0, xb = 0;
  for (long long i = lo; i < hi; ++i) { xa += a[i]; if (b) xb += b[i]; }
  sa[t] = xa; sb[t] = xb;
  __syncthreads();
  // Hillis-Steele inclusive scan over 1024 partials
  for (int o = 1; o < 1024; o <<= 1) {
    uint32_t ya = 0, yb = 0;
    if (t >= o) { ya = sa[t - o]; yb = sb[t - o]; }
    __syncthreads();
    sa[t] += ya; sb[t] += yb;
    __syncthreads();
  }
  uint32_t ra = sa[t] - xa, rb = sb[t] - xb;  // exclusive base of this thread's chunk
  for (long long i = lo; i < hi; ++i) {
    const uint32_t va = a[i]; a[i] = ra; ra += va;
    if (b) { const uint32_t vb = b[i]; b[i] = rb; rb += vb; }
  }
}

// ---- multi-block exclusive scan: local scans of 8192-entry chunks, scan of the chunk totals, fix-up ----
constexpr int SCAN_CHUNK = 8192;

__global__ void __launch_bounds__(1024)
scan_local_kernel(uint32_t *a, uint32_t *b, long long n, uint32_t *tot_a, uint32_t *tot_b) {
  __shared__ uint32_t wa[32], wb[32];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const long long base = (long long)blockIdx.x * SCAN_CHUNK + (long long)t * 8;
  uint32_t va[8], vb[8];
  uint32_t sa = 0, sb = 0;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const long long i = base + q;
    va[q] = i < n ? a[i] : 0u;
    vb[q] = (b && i < n) ? b[i] : 0u;
    sa += va[q]; sb += vb[q];
  }
  uint32_t ia = sa, ib = sb;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t ya = __shfl_up_sync(FULL, ia, d), yb = __shfl_up_sync(FULL, ib, d);
    if (lane >= d) { ia += ya; ib += yb; }
  }
  if (lane == 31) { wa[warp] = ia; wb[warp] = ib; }
  __syncthreads();
  if (warp == 0) {
    uint32_t xa = wa[lane], xb = wb[lane];
    uint32_t ja = xa, jb = xb;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t ya = __shfl_up_sync(FULL, ja, d), yb = __shfl_up_sync(FULL, jb, d);
      if (lane >= d) { ja += ya; jb += yb; }
    }
    wa[lane] = ja - xa; wb[lane] = jb - xb;
    if (lane == 31) { tot_a[blockIdx.x] = ja; if (b) tot_b[blockIdx.x] = jb; }
  }
  __syncthreads();
  uint32_t ra = wa[warp] + ia - sa, rb = wb[warp] + ib - sb;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const long long i = base + q;
    if (i < n) {
      a[i] = ra; ra += va[q];
      if (b) { b[i] = rb; rb += vb[q]; }
    }
  }
}

__global__ void __launch_bounds__(1024)
scan_fixup_kernel(uint32_t *a, uint32_t *b, long long n, const uint32_t *tot_a, const uint32_t *tot_b) {
  const long long base = (long long)blockIdx.x * SCAN_CHUNK;
  const uint32_t oa = tot_a[blockIdx.x], ob = b ? tot_b[blockIdx.x] : 0u;
  for (int t = threadIdx.x; t < SCAN_CHUNK; t += 1024) {
    const long long i = base + t;
    if (i < n) { a[i] += oa; if (b) b[i] += ob; }
  }
}

// exclusive scan of a (and b) in place; tmp holds 2 * ceil(n / SCAN_CHUNK) uint32
static void scan_exclusive(uint32_t *a, uint32_t *b, long long n, uint32_t *tmp, cudaStream_t stream) {
  if (n <= SCAN_CHUNK) {
    scan_exclusive_kernel<<<1, 1024, 0, stream>>>(a, b, n);
    return;
  }
  const int nchunks = (int)((n + SCAN_CHUNK - 1) / SCAN_CHUNK);
  uint32_t *ta = tmp, *tb = tmp + nchunks;
  scan_local_kernel<<<nchunks, 1024, 0, stream>>>(a, b, n, ta, tb);
  scan_exclusive_kernel<<<1, 1024, 0, stream>>>(ta, b ? tb : nullptr, (long long)nchunks);
  scan_fixup_kernel<<<nchunks, 1024, 0, stream>>>(a, b, n, ta, tb);
}

__global__ void __launch_bounds__(TK_THREADS)
topk_write_kernel(const ScoreSrc score, long long M, const TopkState *state,
                  const uint32_t *__restrict__ blk_less, const uint32_t *__restrict__ blk_eq,
                  uint32_t *__restrict__ out_key, uint32_t *__restrict__ out_idx) {
  const uint32_t T = state->prefix;
  const uint32_t r = state->need_eq;
  const long long base = (long long)blockIdx.x * TK_TILE;
  uint32_t run_less = blk_less[blockIdx.x];  // global #less before the current sub-chunk
  uint32_t run_eq = blk_eq[blockIdx.x];      // global #eq   before the current sub-chunk
  __shared__ uint32_t wsum[TK_THREADS / 32];
  __shared__ uint32_t s_tot;
  const int lane = lane_id(), warp = threadIdx.x >> 5;
  // sub-chunk: 4 consecutive elements per thread, 1024 per block iteration
  for (int sub = 0; sub < TK_TILE; sub += TK_THREADS * 4) {
    const long long i0 = base + sub + (long long)threadIdx.x * 4;
    uint32_t key[4];
    uint32_t cls[4];  // 1 = less, 0x10000 = eq
    uint32_t mine = 0;
    float v4[4];
    score.load4(i0, M, v4);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const long long i = i0 + q;
      key[q] = 0; cls[q] = 0;
      if (i < M) {
        key[q] = score_key(v4[q]);
        cls[q] = key[q] < T ? 1u : (key[q] == T ? 0x10000u : 0u);
      }
      mine += cls[q];
    }
    // packed (less | eq<<16) exclusive block scan; both fields <= 1024
    uint32_t inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(FULL, inc, d);
      if (lane >= d) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t acc = 0;
      for (int w = 0; w < TK_THREADS / 32; ++w) { uint32_t v = wsum[w]; wsum[w] = acc; acc += v; }
      s_tot = acc;
    }
    __syncthreads();
    uint32_t ex = wsum[warp] + inc - mine;
    uint32_t lb = run_less + (ex & 0xffffu);
    uint32_t eb = run_eq + (ex >> 16);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (cls[q] == 1u) {
        const uint32_t pos = lb + min(eb, r);
        out_key[pos] = key[q];
        out_idx[pos] = (uint32_t)(i0 + q);
        lb++;
      } else if (cls[q] == 0x10000u) {
        if (eb < r) {
          const uint32_t pos = lb + eb;
          out_key[pos] = key[q];
          out_idx[pos] = (uint32_t)(i0 + q);
        }
        eb++;
      }
    }
    const uint32_t tot = s_tot;
    run_less += tot & 0xffffu;
    run_eq += tot >> 16;
    __syncthreads();
  }
}

// ---------------- stable LSD radix sort of (key, idx) by key, 8 bits per pass ----------------

__global__ void __launch_bounds__(TK_THREADS)
sort_hist_kernel(const uint32_t *__restrict__ key, uint32_t k, int shift, uint32_t nb,
                 uint32_t *__restrict__ table /*[256][nb]*/) {
  __shared__ uint32_t sh[256];
  sh[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t base = blockIdx.x * SORT_TILE;
  for (int t = threadIdx.x; t < SORT_TILE; t += TK_THREADS) {
    const uint32_t i = base + t;
    if (i < k) atomicAdd(&sh[(key[i] >> shift) & 255u], 1u);
  }
  __syncthreads();
  table[(size_t)threadIdx.x * nb + blockIdx.x] = sh[threadIdx.x];
}

__global__ void __launch_bounds__(TK_THREADS)
sort_scatter_kernel(const uint32_t *__restrict__ key_in, const uint32_t *__restrict__ idx_in,
                    uint32_t k, int shift, uint32_t nb, const uint32_t *__restrict__ table,
                    uint32_t *__restrict__ key_out, uint32_t *__restrict__ idx_out) {
  __shared__ uint32_t warp_cnt[TK_THREADS / 32][256];
  __shared__ uint32_t digit_base[256];
  const int tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
  digit_base[tid] = table[(size_t)tid * nb + blockIdx.x];
  const uint32_t base = blockIdx.x * SORT_TILE;
  for (int sub = 0; sub < SORT_TILE; sub += TK_THREADS) {
#pragma unroll
    for (int w = 0; w < TK_THREADS / 32; ++w) warp_cnt[w][tid] = 0;
    __syncthreads();
    const uint32_t i = base + sub + tid;
    const bool valid = i < k;
    uint32_t kk = 0, ii = 0;
    if (valid) { kk = key_in[i]; ii = idx_in[i]; }
    const uint32_t d = valid ? ((kk >> shift) & 255u) : (0x100u | lane);
    const unsigned peers = __match_any_sync(FULL, d);
    const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
    if (valid && rank == 0) warp_cnt[warp][d] = __popc(peers);
    __syncthreads();
    uint32_t run = 0;
#pragma unroll
    for (int w = 0; w < TK_THREADS / 32; ++w) {
      const uint32_t c = warp_cnt[w][tid];
      warp_cnt[w][tid] = run;
      run += c;
    }
    __syncthreads();
    if (valid) {
      const uint32_t pos = digit_base[d] + warp_cnt[warp][d] + rank;
      key_out[pos] = kk;
      idx_out[pos] = ii;
    }
    __syncthreads();
    digit_base[tid] += run;
  }
}

__global__ void topk_finalize_kernel(const ScoreSrc score,
                                     const uint32_t *__restrict__ idx, uint32_t k,
                                     uint32_t *__restrict__ out_idx, float *__restrict__ out_score) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < k) {
    const uint32_t p = idx[i];
    if (out_idx) out_idx[i] = p;
    if (out_score) out_score[i] = score.at(p);
  }
}

// (u, v) of virtual position p: segment A (the running list) first, then segment B (the slab)
__global__ void gather_pairs2_kernel(const int *__restrict__ ua, const int *__restrict__ va, long long na,
                                     const int *__restrict__ ub, const int *__restrict__ vb,
                                     const uint32_t *__restrict__ idx, long long k,
                                     int *__restrict__ out_u, int *__restrict__ out_v) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < k) {
    const long long p = idx[i];
    if (p < na) { out_u[i] = ua[p]; out_v[i] = va[p]; }
    else        { out_u[i] = ub[p - na]; out_v[i] = vb[p - na]; }
  }
}

__global__ void pack_edges_kernel(const int *__restrict__ pu, const int *__restrict__ pv,
                                  const uint32_t *__restrict__ idx, const float *__restrict__ score,
                                  long long k, float *__restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < k) {
    const uint32_t p = idx ? idx[i] : (uint32_t)i;
    out[i * 3 + 0] = (float)pu[p];
    out[i * 3 + 1] = (float)pv[p];
    out[i * 3 + 2] = score[i];
  }
}


// ---------------- K4b: threshold push-down (ordered compaction under the running k-th score) ----------------
// Once a running proposal list holds k candidates, a new slab can only contribute elements that beat the
// list's k-th score s_k: strictly (a tie at s_k loses to the list's own ties, which come earlier in candidate
// order), or — prefilter mode, scores later re-computed in fp32 — everything with score >= s_k - margin.
// One counting read and one writing read of the slab's scores replace five radix-select reads of it; the
// survivors keep their position order, so the tie rule needs nothing else.

__device__ __forceinline__ float key_score(uint32_t key) {
  const uint32_t asc = ~key;
  const uint32_t b = (asc >> 31) ? (asc ^ 0x80000000u) : ~asc;
  return __uint_as_float(b);
}

// largest key that still survives (keys ascend as scores descend)
__device__ __forceinline__ uint32_t threshold_last_key(uint32_t bound, float margin, int inclusive) {
  if (!inclusive) return bound == 0 ? 0u : bound - 1;       // strictly better than the k-th (bound 0: nothing can be)
  if (!(margin > 0.f)) return bound;
  const uint32_t kt = score_key(key_score(bound) - margin);
  return kt == 0xffffffffu ? kt : kt + 1;                   // one ulp of slack below the rounded difference
}

__global__ void __launch_bounds__(TK_THREADS)
threshold_count_kernel(const float *__restrict__ score, long long M, const uint32_t *__restrict__ bound_key,
                       float margin, int inclusive, uint32_t *__restrict__ tile_count) {
  const uint32_t bound = *bound_key;
  const bool none = !inclusive && bound == 0;
  const uint32_t last = threshold_last_key(bound, margin, inclusive);
  const ScoreSrc src{nullptr, 0, score};
  const long long base = (long long)blockIdx.x * TK_TILE;
  uint32_t c = 0;
#pragma unroll
  for (int t = 0; t < TK_TILE; t += TK_THREADS * 4) {
    const long long i = base + t + threadIdx.x * 4;
    float v[4];
    src.load4(i, M, v);
#pragma unroll
    for (int q = 0; q < 4; ++q) c += (i + q < M && !none && score_key(v[q]) <= last);
  }
  __shared__ uint32_t sc[TK_THREADS / 32];
#pragma unroll
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(FULL, c, o);
  if (lane_id() == 0) sc[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t a = 0;
    for (int w = 0; w < TK_THREADS / 32; ++w) a += sc[w];
    tile_count[blockIdx.x] = a;
    if (blockIdx.x == 0) tile_count[gridDim.x] = 0;       // slot of the grand total (exclusive scan)
  }
}

__global__ void __launch_bounds__(TK_THREADS)
threshold_write_kernel(const float *__restrict__ score, const int *__restrict__ pu, const int *__restrict__ pv,
                       long long M, const uint32_t *__restrict__ bound_key, float margin, int inclusive,
                       const uint32_t *__restrict__ tile_off, int *__restrict__ out_u, int *__restrict__ out_v,
                       float *__restrict__ out_score, uint32_t *__restrict__ out_pos) {
  const uint32_t bound = *bound_key;
  const bool none = !inclusive && bound == 0;
  const uint32_t last = threshold_last_key(bound, margin, inclusive);
  if (tile_off[blockIdx.x + 1] == tile_off[blockIdx.x]) return;   // nothing survives in this tile
  const ScoreSrc src{nullptr, 0, score};
  const long long base = (long long)blockIdx.x * TK_TILE;
  uint32_t run = tile_off[blockIdx.x];
  __shared__ uint32_t wsum[TK_THREADS / 32];
  __shared__ uint32_t s_tot;
  const int lane = lane_id(), warp = threadIdx.x >> 5;
  for (int sub = 0; sub < TK_TILE; sub += TK_THREADS * 4) {
    const long long i0 = base + sub + (long long)threadIdx.x * 4;
    float v4[4];
    src.load4(i0, M, v4);
    bool ok[4];
    uint32_t mine = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      ok[q] = i0 + q < M && !none && score_key(v4[q]) <= last;
      mine += ok[q];
    }
    uint32_t inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t t = __shfl_up_sync(FULL, inc, d);
      if (lane >= d) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t acc = 0;
      for (int w = 0; w < TK_THREADS / 32; ++w) { const uint32_t v = wsum[w]; wsum[w] = acc; acc += v; }
      s_tot = acc;
    }
    __syncthreads();
    uint32_t pos = run + wsum[warp] + inc - mine;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (ok[q]) {
        if (out_u) { out_u[pos] = pu[i0 + q]; out_v[pos] = pv[i0 + q]; }
        if (out_score) out_score[pos] = v4[q];
        if (out_pos) out_pos[pos] = (uint32_t)(i0 + q);
        ++pos;
      }
    }
    run += s_tot;
    __syncthreads();
  }
}

static inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct TopkLayout {
  size_t state, hist, blk_less, blk_eq, keyA, keyB, idxA, idxB, table, scan_tmp, total;
  uint32_t nblk, nb_sort;
};

static TopkLayout topk_layout(int64_t M, int64_t k) {
  TopkLayout L;
  L.nblk = (uint32_t)((M + TK_TILE - 1) / TK_TILE);
  L.nb_sort = (uint32_t)((k + SORT_TILE - 1) / SORT_TILE);
  size_t o = 0;
  L.state = o; o += 256;
  L.hist = o; o += align256(3 * 2048 * sizeof(uint32_t));
  L.blk_less = o; o += align256((size_t)L.nblk * 4);
  L.blk_eq = o; o += align256((size_t)L.nblk * 4);
  L.keyA = o; o += align256((size_t)k * 4);
  L.keyB = o; o += align256((size_t)k * 4);
  L.idxA = o; o += align256((size_t)k * 4);
  L.idxB = o; o += align256((size_t)k * 4);
  L.table = o; o += align256((size_t)256 * L.nb_sort * 4);
  const size_t longest = std::max<size_t>(L.nblk, (size_t)256 * L.nb_sort);
  L.scan_tmp = o; o += align256(2 * ((longest + SCAN_CHUNK - 1) / SCAN_CHUNK + 1) * 4);
  L.total = o;
  return L;
}

}  // namespace eps

extern "C" size_t eps_topk_workspace_bytes(int64_t M, int64_t k) {
  if (M <= 0 || k <= 0) return 256;
  return eps::topk_layout(M, k).total;
}

namespace eps {
// steps 1-3 (+ 4 when `sorted`) over the concatenation src = A ++ B of M elements
static int topk_run(const ScoreSrc src, int64_t M, int64_t k, bool sorted, const uint32_t *prune_key,
                    uint32_t *kth_key_out, uint32_t *out_idx, float *out_score,
                    void *workspace, size_t workspace_bytes, cudaStream_t stream, const char *who) {
  const int sms = sm_count();
  if (sms <= 0) { set_error("%s: no CUDA device", who); return EPS_ERR_CUDA; }
  const TopkLayout L = topk_layout(M, k);
  if (!workspace || workspace_bytes < L.total) {
    set_error("%s: workspace too small (%zu < %zu)", who, workspace_bytes, L.total);
    return EPS_ERR_WORKSPACE;
  }
  char *ws = (char *)workspace;
  TopkState *state = (TopkState *)(ws + L.state);
  uint32_t *hist = (uint32_t *)(ws + L.hist);
  uint32_t *blk_less = (uint32_t *)(ws + L.blk_less), *blk_eq = (uint32_t *)(ws + L.blk_eq);
  uint32_t *keyA = (uint32_t *)(ws + L.keyA), *keyB = (uint32_t *)(ws + L.keyB);
  uint32_t *idxA = (uint32_t *)(ws + L.idxA), *idxB = (uint32_t *)(ws + L.idxB);
  uint32_t *table = (uint32_t *)(ws + L.table);
  uint32_t *scan_tmp = (uint32_t *)(ws + L.scan_tmp);

  EPS_CUDA(cudaMemsetAsync(ws + L.state, 0, L.blk_less - L.state, stream));  // state + hist
  const long long want = (M + TK_THREADS * 8 - 1) / (TK_THREADS * 8);
  const int hgrid = (int)std::max<long long>(1, std::min<long long>(want, (long long)sms * 8));
  topk_hist_kernel<0><<<hgrid, TK_THREADS, 0, stream>>>(src, M, state, prune_key, hist);
  topk_pick_kernel<0><<<1, 256, 0, stream>>>(state, hist, (uint32_t)k, nullptr);
  topk_hist_kernel<1><<<hgrid, TK_THREADS, 0, stream>>>(src, M, state, nullptr, hist + 2048);
  topk_pick_kernel<1><<<1, 256, 0, stream>>>(state, hist + 2048, (uint32_t)k, nullptr);
  topk_hist_kernel<2><<<hgrid, TK_THREADS, 0, stream>>>(src, M, state, nullptr, hist + 4096);
  topk_pick_kernel<2><<<1, 256, 0, stream>>>(state, hist + 4096, (uint32_t)k, kth_key_out);
  EPS_LAUNCH_CHECK();
  if (!out_idx && !out_score) return EPS_OK;          // only the k-th key was asked for
  topk_count_kernel<<<L.nblk, TK_THREADS, 0, stream>>>(src, M, state, blk_less, blk_eq);
  scan_exclusive(blk_less, blk_eq, (long long)L.nblk, scan_tmp, stream);
  topk_write_kernel<<<L.nblk, TK_THREADS, 0, stream>>>(src, M, state, blk_less, blk_eq, keyA, idxA);
  EPS_LAUNCH_CHECK();
  uint32_t *kin = keyA, *iin = idxA, *kout = keyB, *iout = idxB;
  for (int pass = 0; sorted && pass < 4; ++pass) {
    const int shift = pass * 8;
    sort_hist_kernel<<<L.nb_sort, TK_THREADS, 0, stream>>>(kin, (uint32_t)k, shift, L.nb_sort, table);
    scan_exclusive(table, nullptr, (long long)256 * L.nb_sort, scan_tmp, stream);
    sort_scatter_kernel<<<L.nb_sort, TK_THREADS, 0, stream>>>(kin, iin, (uint32_t)k, shift, L.nb_sort,
                                                              table, kout, iout);
    std::swap(kin, kout);
    std::swap(iin, iout);
  }
  EPS_LAUNCH_CHECK();
  topk_finalize_kernel<<<(unsigned)((k + 255) / 256), 256, 0, stream>>>(src, iin, (uint32_t)k, out_idx, out_score);
  EPS_LAUNCH_CHECK();
  return EPS_OK;
}
}  // namespace eps

extern "C" int eps_topk_f32(const float *score, int64_t M, int64_t k, uint32_t *out_idx,
                            float *out_score, void *workspace, size_t workspace_bytes,
                            void *stream_) {
  using namespace eps;
  EPS_CHECK_ARG(score != nullptr, "score is NULL");
  EPS_CHECK_ARG(out_idx || out_score, "no output requested");
  EPS_CHECK_ARG(M >= 1 && M < 0xffffffffll, "M out of range [1, 2^32-1)");
  EPS_CHECK_ARG(k >= 1 && k <= M, "k out of range [1, M]");
  return topk_run(ScoreSrc{nullptr, 0, score}, M, k, true, nullptr, nullptr, out_idx, out_score, workspace,
                  workspace_bytes, (cudaStream_t)stream_, "eps_topk_f32");
}

extern "C" int eps_topk_select2_f32(const float *score_a, int64_t Ma, const float *score_b, int64_t Mb,
                                    int64_t k, const uint32_t *prune_key, uint32_t *kth_key_out,
                                    uint32_t *out_idx, float *out_score, void *workspace,
                                    size_t workspace_bytes, void *stream_) {
  using namespace eps;
  EPS_CHECK_ARG(Ma >= 0 && Mb >= 0 && (Ma == 0 || score_a) && (Mb == 0 || score_b), "bad segments");
  EPS_CHECK_ARG(out_idx || out_score || kth_key_out, "no output requested");
  const int64_t M = Ma + Mb;
  EPS_CHECK_ARG(M >= 1 && M < 0xffffffffll, "Ma + Mb out of range [1, 2^32-1)");
  EPS_CHECK_ARG(k >= 1 && k <= M, "k out of range [1, Ma + Mb]");
  return topk_run(ScoreSrc{score_a, Ma, score_b}, M, k, false, prune_key, kth_key_out, out_idx, out_score,
                  workspace, workspace_bytes, (cudaStream_t)stream_, "eps_topk_select2_f32");
}


extern "C" int64_t eps_threshold_tiles(int64_t M) { return M <= 0 ? 0 : (M + eps::TK_TILE - 1) / eps::TK_TILE; }

extern "C" int eps_threshold_count(const float *score, int64_t M, const uint32_t *bound_key, float margin,
                                   int inclusive, uint32_t *tile_offsets, void *workspace,
                                   size_t workspace_bytes, void *stream_) {
  using namespace eps;
  EPS_CHECK_ARG(M >= 0 && M < 0xffffffffll, "M out of range [0, 2^32-1)");
  EPS_CHECK_ARG(bound_key && tile_offsets, "null pointer");
  EPS_CHECK_ARG(margin >= 0.f, "negative margin");
  cudaStream_t stream = (cudaStream_t)stream_;
  if (M == 0) { EPS_CUDA(cudaMemsetAsync(tile_offsets, 0, 4, stream)); return EPS_OK; }
  EPS_CHECK_ARG(score != nullptr, "score is NULL");
  if (sm_count() <= 0) { set_error("eps_threshold_count: no CUDA device"); return EPS_ERR_CUDA; }
  const long long nt = (M + TK_TILE - 1) / TK_TILE;
  const size_t need = align256(2 * ((size_t)(nt + 1 + SCAN_CHUNK - 1) / SCAN_CHUNK + 1) * 4);
  if (!workspace || workspace_bytes < need) {
    set_error("eps_threshold_count: workspace too small (%zu < %zu)", workspace_bytes, need);
    return EPS_ERR_WORKSPACE;
  }
  threshold_count_kernel<<<(unsigned)nt, TK_THREADS, 0, stream>>>(score, M, bound_key, margin, inclusive, tile_offsets);
  scan_exclusive(tile_offsets, nullptr, nt + 1, (uint32_t *)workspace, stream);
  EPS_LAUNCH_CHECK();
  return EPS_OK;
}

extern "C" size_t eps_threshold_workspace_bytes(int64_t M) {
  const long long nt = M <= 0 ? 0 : (M + eps::TK_TILE - 1) / eps::TK_TILE;
  return eps::align256(2 * ((size_t)(nt + 1 + eps::SCAN_CHUNK - 1) / eps::SCAN_CHUNK + 1) * 4) + 256;
}

extern "C" int eps_threshold_write(const float *score, const int32_t *pair_u, const int32_t *pair_v, int64_t M,
                                   const uint32_t *bound_key, float margin, int inclusive,
                                   const uint32_t *tile_offsets, int32_t *out_u, int32_t *out_v,
                                   float *out_score, uint32_t *out_pos, void *stream_) {
  using namespace eps;
  EPS_CHECK_ARG(M >= 0 && M < 0xffffffffll, "M out of range [0, 2^32-1)");
  if (M == 0) return EPS_OK;
  EPS_CHECK_ARG(score && bound_key && tile_offsets, "null pointer");
  EPS_CHECK_ARG((out_u != nullptr) == (out_v != nullptr), "out_u and out_v come together");
  EPS_CHECK_ARG(!out_u || (pair_u && pair_v), "pairs requested without pair_u / pair_v");
  EPS_CHECK_ARG(out_u || out_score || out_pos, "no output requested");
  const long long nt = (M + TK_TILE - 1) / TK_TILE;
  threshold_write_kernel<<<(unsigned)nt, TK_THREADS, 0, (cudaStream_t)stream_>>>(
      score, pair_u, pair_v, M, bound_key, margin, inclusive, tile_offsets, out_u, out_v, out_score, out_pos);
  EPS_LAUNCH_CHECK();
  return EPS_OK;
}

extern "C" int eps_gather_pairs2(const int32_t *ua, const int32_t *va, int64_t Ma, const int32_t *ub,
                                 const int32_t *vb, const uint32_t *idx, int64_t k, int32_t *out_u,
                                 int32_t *out_v, void *stream_) {
  using namespace eps;
  EPS_CHECK_ARG(idx && out_u && out_v && Ma >= 0 && k >= 0, "null pointer or negative size");
  EPS_CHECK_ARG(Ma == 0 || (ua && va), "segment A is NULL");
  if (k == 0) return EPS_OK;
  gather_pairs2_kernel<<<(unsigned)((k + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(
      ua, va, (long long)Ma, ub, vb, idx, (long long)k, out_u, out_v);
  EPS_LAUNCH_CHECK();
  return EPS_OK;
}

extern "C" int eps_pack_edges(const int32_t *pair_u, const int32_t *pair_v, const uint32_t *idx,
                              const float *score, int64_t k, float *out_k3, void *stream_) {
  using namespace eps;
  EPS_CHECK_ARG(pair_u && pair_v && score && out_k3, "null pointer");
  EPS_CHECK_ARG(k >= 0, "negative k");
  if (k == 0) return EPS_OK;
  pack_edges_kernel<<<(unsigned)((k + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(
      pair_u, pair_v, idx, score, (long long)k, out_k3);
  EPS_LAUNCH_CHECK();
  return EPS_OK;
}


// ---------------- K4c: segmented top-m select over owner slabs (per-node proposal budgets) ----------------
// Segments are the owners of a slab: offsets[s] .. offsets[s+1] of the candidate list, contiguous and in candidate
// order.  Per segment, the same three radix passes as K4 (11+11+10 bits, same keys, same tie rule) find the m-th key
// T and r = how many elements equal to T are still needed; the write pass is K4's ordered compaction restricted to
// the segment.  Band mode keeps every element whose key is <= threshold_last_key(T, margin, inclusive) — the bound of
// K4b, so both prefilter paths round the same way.
//   select: persistent CTAs take segments from a list with the large ones first (a hub left for last would be the tail
//           of the launch); a segment of <= m elements passes through without a histogram, one of <= SEG_SMEM_KEYS
//           keys is loaded into shared memory once, larger ones are streamed from L2 / HBM by every pass.
//   scan:   the per-segment kept counts -> output offsets (the last entry is the survivor count the host reads).
//   write:  persistent CTAs again; each copies its segment's survivors (u, v, score) in position order.
namespace eps {

constexpr int SEG_THREADS = 256;
constexpr int SEG_SMEM_KEYS = 6144;          // 24 KB of keys next to the 8 KB histogram
constexpr long long SEG_BIG = 16384;         // segments above this go to the front of the work list

struct SegCtl {
  uint32_t n_big, n_small, next_select, next_write;
};

__device__ __forceinline__ void seg_bounds(const long long *__restrict__ off, long long s, long long M,
                                           long long &lo, long long &hi) {
  lo = min(max(off[s], 0ll), M);
  hi = min(max(off[s + 1], lo), M);
}

// work list: segments larger than SEG_BIG at the front, the others behind them (order inside a group is irrelevant:
// every segment's result depends on its own elements only)
__global__ void seg_order_kernel(const long long *__restrict__ off, long long n_seg, long long M, SegCtl *ctl,
                                 uint32_t *__restrict__ order) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_seg) return;
  long long lo, hi;
  seg_bounds(off, s, M, lo, hi);
  if (hi - lo > SEG_BIG) order[atomicAdd(&ctl->n_big, 1u)] = (uint32_t)s;
  else order[n_seg - 1 - atomicAdd(&ctl->n_small, 1u)] = (uint32_t)s;
}

// one 256-thread block: the bin d of hist[NB] that holds the k_rem-th element (1-based) and cum = #elements in the
// bins below d (topk_pick_kernel's search, inside the CTA that built the histogram)
template <int NB>
__device__ __forceinline__ void seg_pick(const uint32_t *hist, uint32_t k_rem, uint32_t *wtot, uint32_t *s_pick) {
  constexpr int PER = NB / SEG_THREADS;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  uint32_t c[PER], mine = 0;
#pragma unroll
  for (int q = 0; q < PER; ++q) { c[q] = hist[t * PER + q]; mine += c[q]; }
  uint32_t inc = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(FULL, inc, d);
    if (lane >= d) inc += y;
  }
  if (lane == 31) wtot[warp] = inc;
  __syncthreads();
  uint32_t base = 0;
  for (int w = 0; w < warp; ++w) base += wtot[w];
  const uint32_t before = base + inc - mine;
  if (before < k_rem && k_rem <= before + mine) {
    uint32_t cum = before;
    int q = 0;
    for (; q < PER - 1; ++q) {
      if (cum + c[q] >= k_rem) break;
      cum += c[q];
    }
    s_pick[0] = (uint32_t)(t * PER + q);
    s_pick[1] = cum;
  }
  __syncthreads();
}

// one radix pass over a segment: histogram of the PASS digit of the keys inside the current prefix bucket, then the
// bucket of the k_rem-th key.  Keys come from shared memory (small segments) or from `score` (hubs).
template <int PASS>
__device__ __forceinline__ void seg_pass(const float *__restrict__ seg, const uint32_t *keys_sh, long long n,
                                         uint32_t *hist, uint32_t *wtot, uint32_t *s_pick, uint32_t &prefix,
                                         uint32_t &k_rem) {
  constexpr int NB = (PASS == 2) ? 1024 : 2048;
  constexpr int SHIFT = (PASS == 0) ? 21 : (PASS == 1 ? 10 : 0);
  for (int i = threadIdx.x; i < NB; i += SEG_THREADS) hist[i] = 0;
  __syncthreads();
  const int lane = lane_id();
  for (long long b = 0; b < n; b += SEG_THREADS) {          // warp-uniform trip count
    const long long i = b + threadIdx.x;
    uint32_t key = 0;
    bool ok = false;
    if (i < n) {
      key = keys_sh ? keys_sh[i] : score_key(__ldg(seg + i));
      ok = pass_match<PASS>(key, prefix);
    }
    const unsigned part = __ballot_sync(FULL, ok);
    if (part == 0) continue;
    const uint32_t d = ok ? pass_digit<PASS>(key) : 0x10000u;
    if (__popc(part) <= 8) {
      if (ok) atomicAdd(&hist[d], 1u);
    } else {                                                  // tie-heavy (CN) keys: one atomic per distinct digit
      const unsigned peers = __match_any_sync(FULL, d);
      if (ok && lane == (__ffs(peers) - 1)) atomicAdd(&hist[d], (uint32_t)__popc(peers));
    }
  }
  __syncthreads();
  seg_pick<NB>(hist, k_rem, wtot, s_pick);
  prefix |= s_pick[0] << SHIFT;
  k_rem -= s_pick[1];
  __syncthreads();
}

// per segment: keep-rule (T, r) — keep key < T, and the first r keys == T — and the kept count
__global__ void __launch_bounds__(SEG_THREADS)
seg_select_kernel(const float *__restrict__ score, long long M, const long long *__restrict__ off, long long n_seg,
                  uint32_t m, float margin, int band, SegCtl *ctl, const uint32_t *__restrict__ order,
                  uint32_t *__restrict__ seg_T, uint32_t *__restrict__ seg_r, uint32_t *__restrict__ count) {
  __shared__ uint32_t hist[2048];
  __shared__ uint32_t keys_sh[SEG_SMEM_KEYS];
  __shared__ uint32_t wtot[SEG_THREADS / 32], s_pick[2], s_item, s_cnt;
  for (;;) {
    if (threadIdx.x == 0) s_item = atomicAdd(&ctl->next_select, 1u);
    __syncthreads();
    const uint32_t item = s_item;
    __syncthreads();
    if (item >= n_seg) return;
    const long long s = order[item];
    long long lo, hi;
    seg_bounds(off, s, M, lo, hi);
    const long long n = hi - lo;
    if (n <= (long long)m) {                                  // the whole segment is kept
      if (threadIdx.x == 0) { seg_T[s] = 0xffffffffu; seg_r[s] = 0xffffffffu; count[s] = (uint32_t)n; }
      continue;
    }
    const float *seg = score + lo;
    const uint32_t *ks = nullptr;
    if (n <= SEG_SMEM_KEYS) {
      for (long long i = threadIdx.x; i < n; i += SEG_THREADS) keys_sh[i] = score_key(__ldg(seg + i));
      ks = keys_sh;
      __syncthreads();
    }
    uint32_t prefix = 0, k_rem = m;
    seg_pass<0>(seg, ks, n, hist, wtot, s_pick, prefix, k_rem);
    seg_pass<1>(seg, ks, n, hist, wtot, s_pick, prefix, k_rem);
    seg_pass<2>(seg, ks, n, hist, wtot, s_pick, prefix, k_rem);
    if (!band) {
      if (threadIdx.x == 0) { seg_T[s] = prefix; seg_r[s] = k_rem; count[s] = m; }
      continue;
    }
    const uint32_t last = threshold_last_key(prefix, margin, 1);
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    uint32_t c = 0;
    for (long long i = threadIdx.x; i < n; i += SEG_THREADS)
      c += (ks ? ks[i] : score_key(__ldg(seg + i))) <= last;
#pragma unroll
    for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(FULL, c, o);
    if (lane_id() == 0 && c) atomicAdd(&s_cnt, c);
    __syncthreads();
    if (threadIdx.x == 0) {
      seg_T[s] = last == 0xffffffffu ? last : last + 1;       // key <= last  <=>  key < last + 1
      seg_r[s] = last == 0xffffffffu ? last : 0u;
      count[s] = s_cnt;
    }
  }
}

// per segment: its survivors, in position order, at out_off[s] (K4's ordered compaction inside the segment)
__global__ void __launch_bounds__(SEG_THREADS)
seg_write_kernel(const float *__restrict__ score, const int *__restrict__ pu, const int *__restrict__ pv, long long M,
                 const long long *__restrict__ off, long long n_seg, SegCtl *ctl, const uint32_t *__restrict__ order,
                 const uint32_t *__restrict__ seg_T, const uint32_t *__restrict__ seg_r,
                 const uint32_t *__restrict__ out_off, int *__restrict__ out_u, int *__restrict__ out_v,
                 float *__restrict__ out_score) {
  __shared__ uint32_t wsum[SEG_THREADS / 32];
  __shared__ uint32_t s_tot, s_item;
  const int lane = lane_id(), warp = threadIdx.x >> 5;
  const ScoreSrc src{nullptr, 0, score};
  for (;;) {
    if (threadIdx.x == 0) s_item = atomicAdd(&ctl->next_write, 1u);
    __syncthreads();
    const uint32_t item = s_item;
    __syncthreads();
    if (item >= n_seg) return;
    const long long s = order[item];
    const uint32_t obase = out_off[s];
    if (out_off[s + 1] == obase) continue;
    long long lo, hi;
    seg_bounds(off, s, M, lo, hi);
    const uint32_t T = seg_T[s], r = seg_r[s];
    uint32_t run_less = 0, run_eq = 0;
    for (long long sub = lo; sub < hi; sub += SEG_THREADS * 4) {
      const long long i0 = sub + (long long)threadIdx.x * 4;
      float v4[4];
      src.load4(i0, hi, v4);
      uint32_t cls[4], mine = 0;                              // 1 = less, 0x10000 = eq
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        cls[q] = 0;
        if (i0 + q < hi) {
          const uint32_t key = score_key(v4[q]);
          cls[q] = key < T ? 1u : (key == T ? 0x10000u : 0u);
        }
        mine += cls[q];
      }
      uint32_t inc = mine;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, inc, d);
        if (lane >= d) inc += t;
      }
      if (lane == 31) wsum[warp] = inc;
      __syncthreads();
      if (threadIdx.x == 0) {
        uint32_t acc = 0;
        for (int w = 0; w < SEG_THREADS / 32; ++w) { const uint32_t v = wsum[w]; wsum[w] = acc; acc += v; }
        s_tot = acc;
      }
      __syncthreads();
      const uint32_t ex = wsum[warp] + inc - mine;
      uint32_t lb = run_less + (ex & 0xffffu), eb = run_eq + (ex >> 16);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        long long pos = -1;
        if (cls[q] == 1u) { pos = lb + min(eb, r); ++lb; }
        else if (cls[q] == 0x10000u) { if (eb < r) pos = lb + eb; ++eb; }
        if (pos >= 0) {
          const long long o = obase + pos;
          out_u[o] = pu[i0 + q];
          out_v[o] = pv[i0 + q];
          out_score[o] = v4[q];
        }
      }
      const uint32_t tot = s_tot;
      run_less += tot & 0xffffu;
      run_eq += tot >> 16;
      __syncthreads();
    }
  }
}

struct SegLayout {
  size_t ctl, order, T, r, scan_tmp, total;
};

static SegLayout seg_layout(int64_t n_seg) {
  SegLayout L;
  const size_t ns = (size_t)std::max<int64_t>(n_seg, 1);
  size_t o = 0;
  L.ctl = o; o += 256;
  L.order = o; o += align256(ns * 4);
  L.T = o; o += align256(ns * 4);
  L.r = o; o += align256(ns * 4);
  L.scan_tmp = o; o += align256(2 * ((ns + 1 + SCAN_CHUNK - 1) / SCAN_CHUNK + 1) * 4);
  L.total = o;
  return L;
}

static int seg_grid(int64_t n_seg) {
  return (int)std::max<long long>(1, std::min<long long>(n_seg, (long long)sm_count() * 4));
}

}  // namespace eps

extern "C" size_t eps_segment_topk_workspace_bytes(int64_t n_seg) {
  return eps::seg_layout(n_seg < 0 ? 0 : n_seg).total;
}

extern "C" int eps_segment_topk_select(const float *score, int64_t M, const int64_t *seg_offsets, int64_t n_seg,
                                       int64_t m, float margin, int band, uint32_t *out_offsets, void *workspace,
                                       size_t workspace_bytes, void *stream_) {
  using namespace eps;
  EPS_CHECK_ARG(M >= 0 && M < 0xffffffffll, "M out of range [0, 2^32-1)");
  EPS_CHECK_ARG(n_seg >= 0 && n_seg < 0xffffffffll, "n_seg out of range [0, 2^32-1)");
  EPS_CHECK_ARG(m >= 1 && m < 0xffffffffll, "m out of range [1, 2^32-1)");
  EPS_CHECK_ARG(out_offsets != nullptr && workspace != nullptr, "null pointer (out_offsets / workspace)");
  EPS_CHECK_ARG(n_seg == 0 || seg_offsets != nullptr, "null pointer (seg_offsets)");
  EPS_CHECK_ARG(M == 0 || score != nullptr, "null pointer (score)");
  EPS_CHECK_ARG(n_seg > 0 || M == 0, "inconsistent offsets: M > 0 elements in no segment");
  EPS_CHECK_ARG(!band || margin >= 0.f, "band mode needs margin >= 0");
  const SegLayout L = seg_layout(n_seg);
  if (workspace_bytes < L.total) {
    set_error("eps_segment_topk_select: workspace too small (%zu < %zu)", workspace_bytes, L.total);
    return EPS_ERR_WORKSPACE;
  }
  cudaStream_t stream = (cudaStream_t)stream_;
  if (sm_count() <= 0) { set_error("eps_segment_topk_select: no CUDA device"); return EPS_ERR_CUDA; }
  char *ws = (char *)workspace;
  SegCtl *ctl = (SegCtl *)(ws + L.ctl);
  uint32_t *order = (uint32_t *)(ws + L.order);
  EPS_CUDA(cudaMemsetAsync(ctl, 0, sizeof(SegCtl), stream));
  EPS_CUDA(cudaMemsetAsync(out_offsets + n_seg, 0, 4, stream));
  if (n_seg == 0) return EPS_OK;
  const long long *off = (const long long *)seg_offsets;
  seg_order_kernel<<<(unsigned)((n_seg + 255) / 256), 256, 0, stream>>>(off, n_seg, M, ctl, order);
  seg_select_kernel<<<seg_grid(n_seg), SEG_THREADS, 0, stream>>>(
      score, M, off, n_seg, (uint32_t)m, margin, band, ctl, order, (uint32_t *)(ws + L.T),
      (uint32_t *)(ws + L.r), out_offsets);
  scan_exclusive(out_offsets, nullptr, n_seg + 1, (uint32_t *)(ws + L.scan_tmp), stream);
  EPS_LAUNCH_CHECK();
  return EPS_OK;
}

extern "C" int eps_segment_topk_write(const float *score, const int32_t *pair_u, const int32_t *pair_v, int64_t M,
                                      const int64_t *seg_offsets, int64_t n_seg, const uint32_t *out_offsets,
                                      int32_t *out_u, int32_t *out_v, float *out_score, void *workspace,
                                      size_t workspace_bytes, void *stream_) {
  using namespace eps;
  EPS_CHECK_ARG(M >= 0 && M < 0xffffffffll, "M out of range [0, 2^32-1)");
  EPS_CHECK_ARG(n_seg >= 0 && n_seg < 0xffffffffll, "n_seg out of range [0, 2^32-1)");
  EPS_CHECK_ARG(n_seg > 0 || M == 0, "inconsistent offsets: M > 0 elements in no segment");
  if (n_seg == 0) return EPS_OK;
  EPS_CHECK_ARG(score && pair_u && pair_v && seg_offsets && out_offsets && workspace, "null pointer (inputs)");
  EPS_CHECK_ARG(out_u && out_v && out_score, "null pointer (outputs)");
  const SegLayout L = seg_layout(n_seg);
  if (workspace_bytes < L.total) {
    set_error("eps_segment_topk_write: workspace too small (%zu < %zu)", workspace_bytes, L.total);
    return EPS_ERR_WORKSPACE;
  }
  cudaStream_t stream = (cudaStream_t)stream_;
  char *ws = (char *)workspace;
  seg_write_kernel<<<seg_grid(n_seg), SEG_THREADS, 0, stream>>>(
      score, pair_u, pair_v, M, (const long long *)seg_offsets, n_seg, (SegCtl *)(ws + L.ctl),
      (const uint32_t *)(ws + L.order), (const uint32_t *)(ws + L.T), (const uint32_t *)(ws + L.r), out_offsets,
      out_u, out_v, out_score);
  EPS_LAUNCH_CHECK();
  return EPS_OK;
}
