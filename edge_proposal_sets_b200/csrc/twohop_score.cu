// K6+K3 fused — 2-hop candidate enumeration WITH Common-Neighbour / Adamic-Adar / RA scores.
//
// Replaces /root/reference/filter.py:96-109 followed by the per-batch scoring loop
// filter.py:113-142 for the heuristic filter models ('simple', 'adamic', 'adamic_ogb',
// 'resource_allocation').  The reference forms A@A to enumerate candidates, THROWS THE VALUES AWAY
// (filter.py:108-109) and then re-derives them pair by pair (models.py:536-554,
// adamic_utils.py:20-23).  But the values are the scores: every 2-path v - k - u contributes one
// common neighbour k to the pair (u, v), so
//     CN(u, v) = #2-paths,      AA / RA (u, v) = sum over the 2-paths of w_k .
// Walking the 2-paths of an owner v costs  sum_{k in N(v)} deg(k)  list elements, whereas scoring
// its candidates one by one (K3) costs  sum_{u in cand(v)} deg(u)  — ~100x more on the ogbl-ppa
// shape (mean CN ~ 1.4, mean degree of a candidate ~ 150).
//
// One CTA per owner v (handed out dynamically, heaviest first), everything in shared memory but the outputs:
//   1. mark     bitmap of U = union of N(k), k in N(v)              (flattened coalesced walk)
//   2. clear    N(v) and v                                           (filter.py:100,103)
//   3. rank     per-word exclusive popcount prefix (u16 inside a 32-word block + u32 per block),
//               and emission of pair_u in ascending u — the reference's column-major order
//   4. score    second walk over the same 2-paths: a set bit u -> rank(u) -> one RED.ADD into the
//               accumulator of that candidate (count as int32, weight as 64-bit fixed point,
//               eps_common.cuh) — integer atomics, hence exact and order-independent
//   5. cleanup  zero the touched bitmap words
// No count pass: every owner writes into a PADDED slot whose offset is the prefix sum of a cheap per-owner upper bound
// (min(#2-paths, n-1-deg), host-side torch ops) and records its real count; a single-block scan turns the counts into
// compact offsets, and the compaction pass — which has to read every accumulator anyway — moves (u, score, count) to the
// compact position, regenerates v from the owner id, and turns the fixed-point sums into fp32 scores (+ sigmoid), or the
// exact counts and the degrees of both ends (two rowptr loads each) into a similarity score (EPS_SCORE_*, after the
// count-only walk).  No inter-CTA dependency.  Results are bit-identical to eps_cn_aa on the same pairs.
// Upper-triangle mode (EPS_TWOHOP_UPPER): only the candidates u > v of owner v.  The candidate relation of a symmetric
// adjacency is symmetric, so this is every unordered pair once; both walks start each N(k) at its lower bound of v + 1
// and the rank / emission / cleanup passes start at the bitmap block that holds v + 1.
#include "eps_common.cuh"

namespace eps {

constexpr int TS_THREADS = 512;   // measured against 1,024 (DESIGN.md, K6+K3 walk groups)
constexpr int TS_LONG = 96;   // lists at least this long are streamed warp-wide without a search
constexpr int TS_DEPTH = 8;   // ... with this many loads in flight per lane (a hub owner's walk is one CTA's latency chain)

// Visit every element of the neighbour lists of N(v).  A warp takes LG lists at a time (LG = 32, 16, ... 1,
// warp-uniform), and the groups are HANDED OUT through a shared-memory counter: with a static round-robin an owner of
// average degree (74 on the ppa shape) gave some warps two groups and the others one, and a warp that drew a hub's
// list kept the other fifteen waiting — 46 % of all stall samples sat at the two barriers behind the walks
// (ncu source counters, profiles/round2_e_twohop.md).  The caller picks the largest LG that still leaves ~4 groups
// per warp to balance with.  `counter` is zero when the walk starts (the caller resets it behind a barrier).
// f.visit(u, p) is called once per 2-path v - k - u (p = index of u in `col`, i.e. inside N(k)) after
// f.select_slot*(lane that holds k's metadata).  Only end points u >= umin are visited: each N(k) is sorted, so its
// walk starts at its lower bound of umin (one binary search per list) and the flattened prefix uses the suffix lengths.
template <typename F>
__device__ __forceinline__ void walk_two_paths(const int *__restrict__ rowptr, const int *__restrict__ col,
                                               int vs, int ve, int lane, int LG, int *counter, int umin, F f) {
  for (;;) {
    int grp = 0;
    if (lane == 0) grp = atomicAdd(counter, 1);
    grp = __shfl_sync(FULL, grp, 0);
    const int base = vs + grp * LG;
    if (base >= ve) break;
    int k = -1, s = 0, len = 0;
    if (lane < LG && base + lane < ve) {
      k = __ldg(col + base + lane);
      s = __ldg(rowptr + k);
      const int e = __ldg(rowptr + k + 1);
      if (umin > 0) {                                  // upper-triangle mode: first position with col >= umin
        int lo = s, hi = e;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (__ldg(col + mid) < umin) lo = mid + 1; else hi = mid;
        }
        s = lo;
      }
      len = e - s;
    }
    f.load_slot(k, base + lane);
    // ---- long lists: the whole warp streams one list, TS_DEPTH loads in flight per lane ----
    unsigned longmask = __ballot_sync(FULL, len >= TS_LONG);
    while (longmask) {
      const int b = __ffs(longmask) - 1;
      longmask &= longmask - 1;
      const int sb = __shfl_sync(FULL, s, b);
      const int lb = __shfl_sync(FULL, len, b);
      f.select_slot(b);
      const int *__restrict__ lp = col + sb;
      for (int off = 0; off < lb; off += 32 * TS_DEPTH) {
        int u[TS_DEPTH];
#pragma unroll
        for (int q = 0; q < TS_DEPTH; ++q) {
          const int p = off + q * 32 + lane;
          u[q] = p < lb ? __ldg(lp + p) : -1;
        }
#pragma unroll
        for (int q = 0; q < TS_DEPTH; ++q)
          if (u[q] >= 0) f.visit(u[q], sb + off + q * 32 + lane);
      }
    }
    // ---- short lists: one flattened sequence ----
    const int slen = len >= TS_LONG ? 0 : len;
    int pin = slen;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      int t = __shfl_up_sync(FULL, pin, d);
      if (lane >= d) pin += t;
    }
    const int pex = pin - slen;
    const int total = __shfl_sync(FULL, pin, 31);
    for (int j = 0; j < total; j += 32) {
      const int p = j + lane;
      int lo = 0;
      for (int step = LG >> 1; step >= 1; step >>= 1) {      // first slot whose inclusive prefix exceeds p
        int t = __shfl_sync(FULL, pin, lo + step - 1);
        if (t <= p) lo += step;
      }
      const int s_t = __shfl_sync(FULL, s, lo);
      const int pe_t = __shfl_sync(FULL, pex, lo);
      f.select_slot_lane(lo);
      if (p < total) f.visit(__ldg(col + s_t + (p - pe_t)), s_t + (p - pe_t));
    }
  }
}

struct MarkVisitor {
  uint32_t *bm, *bm2;
  __device__ __forceinline__ void load_slot(int, int) {}
  __device__ __forceinline__ void select_slot(int) {}
  __device__ __forceinline__ void select_slot_lane(int) {}
  __device__ __forceinline__ void visit(int u, int) {
    const uint32_t bit = 1u << (u & 31);
    const int w = u >> 5;
    if (!(bm[w] & bit)) {                          // cheap pre-test: most bits are already set
      const uint32_t old = atomicOr(&bm[w], bit);
      if (old == 0) atomicOr(&bm2[w >> 5], 1u << (w & 31));
    }
  }
};

// Weighted adjacency (HAS_VAL, collab): the term of the 2-path v - k - u is a_u * (a_v * w_k) (or a_u * a_v
// without a weight table) with a_v = A[v,k] (the value next to k in N(v)) and a_u = A[k,u] (next to u in
// N(k)) — the same fp32 products as eps_cn_aa forms from A[u,k]; the caller guarantees A[k,u] == A[u,k]
// bit for bit (candidates.py checks it once per graph).
template <bool HAS_W, bool WANT_CN, bool HAS_VAL>
struct ScoreVisitor {
  const uint32_t *bm, *blk;
  const uint16_t *pre;
  const float *__restrict__ wtable;
  const float *__restrict__ val;
  unsigned long long *acc;   // + out_base already applied
  int *cn;
  unsigned long long fx_slot = 0ull, fx = 0ull;
  float sv_slot = 0.f, sv = 0.f;
  __device__ __forceinline__ void load_slot(int k, int pos) {
    if (HAS_VAL) {
      const float a_v = k >= 0 ? __ldg(val + pos) : 0.f;
      sv_slot = (HAS_W && k >= 0) ? __fmul_rn(a_v, __ldg(wtable + k)) : a_v;
    } else if (HAS_W) {
      fx_slot = k >= 0 ? to_fixed(__ldg(wtable + k)) : 0ull;
    }
  }
  __device__ __forceinline__ void select_slot(int b) {           // warp-uniform slot
    if (HAS_VAL) sv = __shfl_sync(FULL, sv_slot, b);
    else if (HAS_W) fx = __shfl_sync(FULL, fx_slot, b);
  }
  __device__ __forceinline__ void select_slot_lane(int lo) {     // per-lane slot
    if (HAS_VAL) sv = __shfl_sync(FULL, sv_slot, lo);
    else if (HAS_W) fx = __shfl_sync(FULL, fx_slot, lo);
  }
  __device__ __forceinline__ void visit(int u, int p) {
    const int w = u >> 5, b = u & 31;
    const uint32_t word = bm[w];
    if ((word >> b) & 1u) {
      const uint32_t idx = blk[w >> 5] + pre[w] + __popc(word & ((1u << b) - 1u));
      if (HAS_VAL) atomicAdd(acc + idx, to_fixed(__fmul_rn(__ldg(val + p), sv)));
      else if (HAS_W) atomicAdd(acc + idx, fx);
      if (WANT_CN) atomicAdd(cn + idx, 1);
    }
  }
};

// Rank pass over the bitmap blocks g0 .. W2 - 1, thread t owning block c + t (32 bitmap words): pre[w] = #candidates
// before word w inside its block (u16), blk[g] = #candidates in the blocks g0 .. g - 1 (u32).  *s_carry is zero on
// entry.  Returns the total, behind a barrier.
template <int THREADS>
__device__ __forceinline__ uint32_t rank_blocks(const uint32_t *bm, const uint32_t *bm2, uint32_t *blk, uint16_t *pre,
                                                int g0, int W2, uint32_t *s_scan, uint32_t *s_carry) {
  const int tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
  constexpr int NW = THREADS / 32;
  for (int c = g0; c < W2; c += THREADS) {
    const int g = c + tid;
    const uint32_t m2 = (g < W2) ? bm2[g] : 0u;
    uint32_t cnt = 0;
    {
      uint32_t m = m2;
      while (m) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        const int w = g * 32 + b;
        pre[w] = (uint16_t)cnt;
        cnt += __popc(bm[w]);
      }
    }
    uint32_t inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(FULL, inc, d);
      if (lane >= d) inc += t;
    }
    if (lane == 31) s_scan[warp] = inc;
    __syncthreads();
    uint32_t wbase = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
      const uint32_t x = s_scan[w];
      if (w < warp) wbase += x;
      tot += x;
    }
    const uint32_t carry = *s_carry;
    if (g < W2) blk[g] = carry + wbase + (inc - cnt);
    __syncthreads();
    if (tid == 0) *s_carry = carry + tot;
  }
  __syncthreads();
  return *s_carry;
}

// Zero the bitmap words that bm2 marks in the blocks g0 .. W2 - 1, and those bm2 blocks.
template <int THREADS>
__device__ __forceinline__ void clear_blocks(uint32_t *bm, uint32_t *bm2, int g0, int W2) {
  for (int g = g0 + threadIdx.x; g < W2; g += THREADS) {
    uint32_t m = bm2[g];
    while (m) {
      const int b = __ffs(m) - 1;
      m &= m - 1;
      bm[g * 32 + b] = 0;
    }
    bm2[g] = 0;
  }
}

// n_order and upper sit before acc: the parameter offsets decide which constant loads ptxas merges, and this order keeps
// the instruction sequence the kernel was measured with.
template <bool HAS_W, bool WANT_CN, bool HAS_VAL>
__global__ void __launch_bounds__(TS_THREADS)
twohop_score_kernel(const int *__restrict__ rowptr, const int *__restrict__ col, const float *__restrict__ val,
                    const float *__restrict__ wtable, int n, int v_lo, int v_hi,
                    const long long *__restrict__ offsets, int *__restrict__ pair_u, int n_order, int upper,
                    unsigned long long *__restrict__ acc, int *__restrict__ cn,
                    unsigned int *owner_counter, unsigned int *__restrict__ counts_out,
                    const int *__restrict__ owner_order) {
  extern __shared__ uint32_t sm[];
  const int W = (n + 31) >> 5;       // bitmap words
  const int W2 = (W + 31) >> 5;      // blocks of 32 words
  uint32_t *bm = sm;
  uint32_t *bm2 = bm + W;            // one bit per non-zero bitmap word
  uint32_t *blk = bm2 + W2;          // #candidates before block g
  uint16_t *pre = reinterpret_cast<uint16_t *>(blk + W2);   // #candidates before word w inside its block
  __shared__ int s_owner;
  __shared__ int s_walk;             // next list group of the current walk
  __shared__ uint32_t s_scan[TS_THREADS / 32];
  __shared__ uint32_t s_carry;
  const int tid = threadIdx.x, lane = lane_id();
  constexpr int NW = TS_THREADS / 32;
  for (int w = tid; w < W + W2; w += TS_THREADS) sm[w] = 0;
  for (;;) {
    __syncthreads();
    if (tid == 0) {
      // owners are handed out HEAVIEST FIRST when the caller supplies an order: a hub owner costs ~40 average owners,
      // and drawn late by one CTA it kept the other 295 waiting — SMs were busy 48 % of the kernel's duration
      // (profiles/round2_e_twohop.md)
      const int t = (int)atomicAdd(owner_counter, 1u);
      s_owner = (owner_order && t < n_order) ? v_lo + owner_order[t] : v_lo + t;
      s_walk = 0;
    }
    __syncthreads();
    const int v = s_owner;
    if (v >= v_hi) break;
    const int vs = __ldg(rowptr + v), ve = __ldg(rowptr + v + 1);
    int LG = 32;                                           // lists per group: ~4 groups per warp to balance with
    while (LG > 1 && (ve - vs + LG - 1) / LG < 4 * NW) LG >>= 1;
    const long long out_base = offsets[v - v_lo];
    if (offsets[v - v_lo + 1] == out_base) continue;   // no (room for) candidates (uniform): bitmap untouched
    // upper-triangle mode (EPS_TWOHOP_UPPER): only candidates u > v, so every bit set below lies at or above umin and
    // the rank pass, emission and cleanup start at the block that holds umin
    const int umin = upper ? v + 1 : 0;
    const int g0 = umin >> 10;                         // first block of 32 bitmap words that can hold a mark
    // ---- 1. mark ----
    walk_two_paths(rowptr, col, vs, ve, lane, LG, &s_walk, umin, MarkVisitor{bm, bm2});
    __syncthreads();
    // ---- 2. clear known edges and the diagonal ----
    for (int p = vs + tid; p < ve; p += TS_THREADS) {
      const int k = __ldg(col + p);
      if (k >= umin) atomicAnd(&bm[k >> 5], ~(1u << (k & 31)));
    }
    if (tid == 0 && v >= umin) atomicAnd(&bm[v >> 5], ~(1u << (v & 31)));
    if (tid == 0) { s_carry = 0; s_walk = 0; }        // the first walk is over (barrier above): reset for the second
    __syncthreads();
    // ---- 3a. rank ----
    const uint32_t total = rank_blocks<TS_THREADS>(bm, bm2, blk, pre, g0, W2, s_scan, &s_carry);
    const bool fits = (long long)total <= offsets[v - v_lo + 1] - out_base;
    // padded slot: record the real count (a violated bound poisons N instead of overrunning the slot)
    if (tid == 0) counts_out[v - v_lo] = fits ? total : 0xffffffffu;
    if (!fits) {
      clear_blocks<TS_THREADS>(bm, bm2, g0, W2);
      continue;
    }
    // ---- 3b. emit pair_u in ascending u (v is regenerated by the compaction) ----
    for (int g = g0 + tid; g < W2; g += TS_THREADS) {
      uint32_t m = bm2[g];
      long long o = out_base + blk[g];
      while (m) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        const int w = g * 32 + b;
        uint32_t bits = bm[w];
        while (bits) {
          const int q = __ffs(bits) - 1;
          bits &= bits - 1;
          pair_u[o] = (w << 5) + q;
          ++o;
        }
      }
    }
    // ---- 4. score: second walk, one integer RED per 2-path that lands on a candidate ----
    if (HAS_W || WANT_CN || HAS_VAL) {
      ScoreVisitor<HAS_W, WANT_CN, HAS_VAL> sv{bm, blk, pre, wtable, val,
                                               (HAS_W || HAS_VAL) ? acc + out_base : nullptr,
                                               WANT_CN ? cn + out_base : nullptr};
      walk_two_paths(rowptr, col, vs, ve, lane, LG, &s_walk, umin, sv);
    }
    __syncthreads();
    // ---- 5. cleanup: a block-uniform loop, not clear_blocks, which changes this kernel's instruction sequence ----
    for (int c = g0; c < W2; c += TS_THREADS) {
      const int g = c + tid;
      if (g < W2) {
        uint32_t m = bm2[g];
        while (m) {
          const int b = __ffs(m) - 1;
          m &= m - 1;
          bm[g * 32 + b] = 0;
        }
        bm2[g] = 0;
      }
    }
  }
}

// Owner order for the one-pass kernel, heaviest first: bucket b = 63 - floor(log2(slot size + 1)), so bucket 0 holds the
// largest slots.  PASS 0 counts, PASS 1 turns the 64 counts into bases (one warp pair), PASS 2 scatters (order inside a
// bucket is whatever the atomics give: the outputs do not depend on the order owners are processed in).
template <int PASS>
__global__ void __launch_bounds__(256)
owner_bucket_kernel(const long long *__restrict__ boff, int n_own, unsigned int *__restrict__ buckets, int *__restrict__ order) {
  if (PASS == 1) {
    __shared__ unsigned int c[64];
    const int t = threadIdx.x;
    c[t] = buckets[t];
    __syncthreads();
    if (t == 0) {
      unsigned int run = 0;
      for (int b = 0; b < 64; ++b) { const unsigned int x = c[b]; c[b] = run; run += x; }
    }
    __syncthreads();
    buckets[t] = c[t];
    return;
  }
  const int stride = gridDim.x * blockDim.x;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_own; i += stride) {
    const unsigned long long sz = (unsigned long long)(boff[i + 1] - boff[i]) + 1ull;
    const int b = __clzll((long long)sz);                 // 63 - floor(log2(sz)); sz >= 1
    if (PASS == 0) atomicAdd(&buckets[b], 1u);
    else order[atomicAdd(&buckets[b], 1u)] = i;
  }
}

// single-block exclusive scan of the per-owner counts (uint32 -> int64 offsets[n_own + 1])
__global__ void __launch_bounds__(1024)
owner_scan_kernel(const unsigned int *__restrict__ counts, int n_own, long long *__restrict__ offsets) {
  __shared__ unsigned long long part[1024];
  const int t = threadIdx.x;
  const int per = (n_own + 1023) / 1024;
  const int lo = min(n_own, t * per), hi = min(n_own, lo + per);
  unsigned long long sum = 0;
  for (int i = lo; i < hi; ++i) sum += counts[i];
  part[t] = sum;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    unsigned long long y = 0;
    if (t >= o) y = part[t - o];
    __syncthreads();
    part[t] += y;
    __syncthreads();
  }
  unsigned long long run = part[t] - sum;
  for (int i = lo; i < hi; ++i) { offsets[i] = (long long)run; run += counts[i]; }
  if (t == 1023) offsets[n_own] = (long long)part[1023];
}

// padded slot of owner v -> compact position; fixed-point sums -> fp32 scores on the way (KIND != 0: counts and the
// degrees of u and v -> the similarity score).
// Work is cut by COMPACT position (tiles of CP_TILE candidates), not by owner, so a hub with 10^5
// candidates does not serialise on one CTA; the owner of a position is found by binary search over the
// compact offsets of the (few) owners the tile touches.
constexpr int CP_THREADS = 256, CP_PER = 8, CP_TILE = CP_THREADS * CP_PER;

// The owner of compact position x < end: lo becomes the largest o in [lo, hi) with cmp_off[o] <= x (invariant:
// cmp_off[lo] <= x < cmp_off[hi]).  For x >= end, lo is left as it is.
__device__ __forceinline__ void owner_search(const long long *cmp_off, int &lo, int hi, long long x, long long end) {
  if (x < end) {
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (cmp_off[mid] <= x) lo = mid; else hi = mid;
    }
  }
}

// the owners of the first and last positions of the tile [base, end), for the whole block (a search of its own:
// owner_search's bound test changes the compaction kernels' instructions here)
__device__ __forceinline__ void tile_owners(const long long *__restrict__ cmp_off, int n_own, long long base,
                                            long long end, int *s_lo, int *s_hi) {
  __syncthreads();
  if (threadIdx.x < 2) {
    const long long x = threadIdx.x == 0 ? base : end - 1;
    int lo = 0, hi = n_own;                       // invariant: cmp_off[lo] <= x < cmp_off[hi]
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (cmp_off[mid] <= x) lo = mid; else hi = mid;
    }
    if (threadIdx.x == 0) *s_lo = lo; else *s_hi = lo;
  }
  __syncthreads();
}

template <int KIND>
__global__ void __launch_bounds__(CP_THREADS)
twohop_compact_kernel(const int *__restrict__ rowptr, const long long *__restrict__ pad_off,
                      const long long *__restrict__ cmp_off, int v_lo, int n_own, long long cap, const int *__restrict__ pad_u,
                      const unsigned long long *__restrict__ acc, const int *__restrict__ cn, int flags,
                      int *__restrict__ pair_u, int *__restrict__ pair_v, float *__restrict__ score,
                      int *__restrict__ count) {
  const long long N = cmp_off[n_own];
  if (N > cap) return;     // a violated bound poisoned N: the caller reports it, nothing is moved
  __shared__ int s_lo, s_hi;
  const long long ntiles = (N + CP_TILE - 1) / CP_TILE;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long base = tile * CP_TILE, end = min(base + (long long)CP_TILE, N);
    tile_owners(cmp_off, n_own, base, end, &s_lo, &s_hi);
    const int o_lo = s_lo, o_hi = s_hi;
    long long src[CP_PER];
    int own[CP_PER];
#pragma unroll
    for (int q = 0; q < CP_PER; ++q) {
      const long long i = base + q * CP_THREADS + threadIdx.x;
      int lo = o_lo;
      owner_search(cmp_off, lo, o_hi + 1, i, end);
      own[q] = lo;
      src[q] = i < end ? pad_off[lo] + (i - cmp_off[lo]) : -1;
    }
    int uu[CP_PER], cc[CP_PER];
    unsigned long long aa[CP_PER];
#pragma unroll
    for (int q = 0; q < CP_PER; ++q) {
      uu[q] = 0; cc[q] = 0; aa[q] = 0ull;
      if (src[q] >= 0) {
        uu[q] = pad_u[src[q]];
        if (acc) aa[q] = acc[src[q]];
        if (cn) cc[q] = cn[src[q]];
      }
    }
    int du[CP_PER], dv[CP_PER];      // similarity kinds: deg u, deg v (rowptr is L2-resident)
    if (KIND && score) {
#pragma unroll
      for (int q = 0; q < CP_PER; ++q) {
        du[q] = dv[q] = 0;
        if (src[q] >= 0) {
          const int v = v_lo + own[q];
          du[q] = __ldg(rowptr + uu[q] + 1) - __ldg(rowptr + uu[q]);
          dv[q] = __ldg(rowptr + v + 1) - __ldg(rowptr + v);
        }
      }
    }
#pragma unroll
    for (int q = 0; q < CP_PER; ++q) {
      if (src[q] < 0) continue;
      const long long i = base + q * CP_THREADS + threadIdx.x;
      pair_u[i] = uu[q];
      pair_v[i] = v_lo + own[q];
      if (score) {
        float sc;
        if (KIND) {
          sc = similarity_score<KIND>(cc[q], du[q], dv[q]);
        } else {
          sc = acc ? from_fixed(aa[q]) : (float)cc[q];
          if (flags & EPS_CN_SIGMOID) sc = sigmoidf_ref(sc);
        }
        score[i] = sc;
      }
      if (count) count[i] = cc[q];
    }
  }
}

using CompactKernel = void (*)(const int *, const long long *, const long long *, int, int, long long, const int *,
                               const unsigned long long *, const int *, int, int *, int *, float *, int *);
// index = score_kind(flags): 0 = CN / AA / RA, 1..7 = the similarity kinds
static const CompactKernel kCompactKinds[8] = {
    twohop_compact_kernel<0>, twohop_compact_kernel<1>, twohop_compact_kernel<2>, twohop_compact_kernel<3>,
    twohop_compact_kernel<4>, twohop_compact_kernel<5>, twohop_compact_kernel<6>, twohop_compact_kernel<7>};

// ---------------------------------------------------------------------------------------------
// Local Path index (eps_local_path_onepass, eps_local_path_pairs; include/eps.h)
//   LP(u, v) = c2 + 1e-3 * c3,  c2 = |N(u) & N(v)| = (A^2)_uv,  c3 = (A^3)_uv = sum_{j in N(u)} c2(j, v).
// On a structurally symmetric graph every j in N(u) with c2(j, v) > 0 is a candidate of v or a neighbour k of v (never
// v itself: a candidate u is not adjacent to v), so for a candidate u of owner v
//   c3(u, v) = sum_{j in N(u) & C(v)} c2(j, v)  +  sum_{k in N(u) & N(v)} tri(v, k),     tri(v, k) = |N(v) & N(k)|.
// The fused kernel gets both sums without a pass over all pairs of 3-paths:
//   walks 1-2  the mark / score walks of twohop_score_kernel over ALL candidates of v (walk 3 looks up j < v in upper
//              mode too); the score walk adds 1 to c2 and, for an emitted candidate, tri of the slot's arc (v, k) to c3;
//   walk 3     while the bitmap is still in shared memory, the N(u) lists of the emitted candidates, 32 per warp,
//              flattened as in cn_aa.cu's grouped_batch: a set bit j -> rank(j) -> c2(j, v) (term 1), summed per
//              candidate in registers (segmented warp scan), one plain store per candidate.
// c2 lives in a per-CTA scratch indexed by the full rank; u, c2 and c3 of the emitted candidates in the padded slot.
// All sums are integers (c3 <= nnz < 2^31), the score is formed once in the compaction pass.
// ---------------------------------------------------------------------------------------------
constexpr int LP_THREADS = 512;
constexpr int LP_LONG = 64;     // walk 3: lists at least this long are streamed warp-wide

__device__ __forceinline__ float local_path_score(int c2, int c3) {
  return __double2float_rn(__dadd_rn((double)c2, __dmul_rn(1e-3, (double)c3)));
}

__device__ __forceinline__ uint32_t bitmap_rank(const uint32_t *bm, const uint32_t *blk, const uint16_t *pre, int w, int b) {
  return blk[w >> 5] + pre[w] + __popc(bm[w] & ((1u << b) - 1u));
}

struct LpScoreVisitor {
  const uint32_t *bm, *blk;
  const uint16_t *pre;
  const int *__restrict__ tri;
  int *c2;                 // per-CTA scratch, full rank
  int *c3;                 // padded slot, rank - lo (candidates u >= umin)
  int lo, umin;
  int t_slot = 0, t = 0;
  __device__ __forceinline__ void load_slot(int k, int pos) { t_slot = k >= 0 ? __ldg(tri + pos) : 0; }
  __device__ __forceinline__ void select_slot(int b) { t = __shfl_sync(FULL, t_slot, b); }
  __device__ __forceinline__ void select_slot_lane(int l) { t = __shfl_sync(FULL, t_slot, l); }
  __device__ __forceinline__ void visit(int u, int) {
    const int w = u >> 5, b = u & 31;
    if ((bm[w] >> b) & 1u) {
      const uint32_t idx = bitmap_rank(bm, blk, pre, w, b);
      atomicAdd(c2 + idx, 1);
      if (u >= umin && t) atomicAdd(c3 + (idx - lo), t);
    }
  }
};

// Walk 3 for the emitted candidates e0 .. e0 + cnt - 1 of the current owner (one warp).  c2 values were produced by L2
// atomics of this CTA (possibly over lines an earlier owner left in L1): read with ld.global.cg.
__device__ __forceinline__ void lp_walk3_batch(const int *__restrict__ rowptr, const int *__restrict__ col,
                                               const uint32_t *bm, const uint32_t *blk, const uint16_t *pre,
                                               const int *c2s, int lo, int *su, int *sc2, int *sc3, int e0, int cnt) {
  const int lane = lane_id();
  int s = 0, len = 0;
  if (lane < cnt) {
    const int u = __ldcg(su + e0 + lane);
    s = __ldg(rowptr + u);
    len = __ldg(rowptr + u + 1) - s;
  }
  int acc = 0;
  // ---- long lists, warp-wide, four loads in flight per lane ----
  unsigned longmask = __ballot_sync(FULL, len >= LP_LONG);
  while (longmask) {
    const int b = __ffs(longmask) - 1;
    longmask &= longmask - 1;
    const int sb = __shfl_sync(FULL, s, b);
    const int lb = __shfl_sync(FULL, len, b);
    int part = 0;
    for (int off = 0; off < lb; off += 128) {
      int j[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int p = off + q * 32 + lane;
        j[q] = p < lb ? __ldg(col + sb + p) : -1;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (j[q] >= 0 && ((bm[j[q] >> 5] >> (j[q] & 31)) & 1u))
          part += __ldcg(c2s + bitmap_rank(bm, blk, pre, j[q] >> 5, j[q] & 31));
    }
    part = __reduce_add_sync(FULL, part);
    if (lane == b) acc += part;
  }
  // ---- short lists, one flattened sequence; hits summed per list by a segmented scan ----
  const int slen = len >= LP_LONG ? 0 : len;
  int pin = slen;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int t = __shfl_up_sync(FULL, pin, d);
    if (lane >= d) pin += t;
  }
  const int pex = pin - slen;
  const int total = __shfl_sync(FULL, pin, 31);
  for (int jb = 0; jb < total; jb += 32) {
    const int p = jb + lane;
    int slot = 0;
#pragma unroll
    for (int step = 16; step >= 1; step >>= 1) {
      const int t = __shfl_sync(FULL, pin, slot + step - 1);
      if (t <= p) slot += step;
    }
    const int s_t = __shfl_sync(FULL, s, slot);
    const int pe_t = __shfl_sync(FULL, pex, slot);
    int x = 0;
    if (p < total) {
      const int j = __ldg(col + s_t + (p - pe_t));
      if ((bm[j >> 5] >> (j & 31)) & 1u) x = __ldcg(c2s + bitmap_rank(bm, blk, pre, j >> 5, j & 31));
    }
    if (__ballot_sync(FULL, x != 0) == 0) continue;          // warp-uniform (a candidate has c2 >= 1)
    // inclusive scan inside runs of equal slot (slots ascend with p, so equal ends mean one run)
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(FULL, x, d);
      const int sl = __shfl_up_sync(FULL, slot, d);
      if (lane >= d && sl == slot) x += t;
    }
    const int lo_b = min(max(pex - jb, 0), 32), hi_b = min(max(pin - jb, 0), 32);
    const int t = __shfl_sync(FULL, x, max(hi_b - 1, 0));   // the run of this lane's list ends at hi_b - 1
    if (hi_b > lo_b) acc += t;
  }
  if (lane < cnt) {
    const int e = e0 + lane;
    sc3[e] = __ldcg(sc3 + e) + acc;
    sc2[e] = __ldcg(c2s + lo + e);
  }
}

__global__ void __launch_bounds__(LP_THREADS)
local_path_onepass_kernel(const int *__restrict__ rowptr, const int *__restrict__ col, const int *__restrict__ tri,
                          int n, int v_lo, int v_hi, const long long *__restrict__ offsets, int *pad_u, int *pad_c2,
                          int *pad_c3, int *scratch, long long scratch_cap, unsigned int *owner_counter,
                          unsigned int *__restrict__ counts_out, const int *__restrict__ owner_order, int n_order,
                          int upper) {
  extern __shared__ uint32_t sm[];
  const int W = (n + 31) >> 5;
  const int W2 = (W + 31) >> 5;
  uint32_t *bm = sm;
  uint32_t *bm2 = bm + W;
  uint32_t *blk = bm2 + W2;
  uint16_t *pre = reinterpret_cast<uint16_t *>(blk + W2);
  __shared__ int s_owner, s_walk, s_walk3;
  __shared__ uint32_t s_scan[LP_THREADS / 32];
  __shared__ uint32_t s_carry, s_lo;
  const int tid = threadIdx.x, lane = lane_id();
  constexpr int NW = LP_THREADS / 32;
  int *c2s = scratch + (long long)blockIdx.x * scratch_cap;
  for (int w = tid; w < W + W2; w += LP_THREADS) sm[w] = 0;
  for (;;) {
    __syncthreads();
    if (tid == 0) {
      const int t = (int)atomicAdd(owner_counter, 1u);
      s_owner = (owner_order && t < n_order) ? v_lo + owner_order[t] : v_lo + t;
      s_walk = 0;
      s_walk3 = 0;
    }
    __syncthreads();
    const int v = s_owner;
    if (v >= v_hi) break;
    const int vs = __ldg(rowptr + v), ve = __ldg(rowptr + v + 1);
    int LG = 32;
    while (LG > 1 && (ve - vs + LG - 1) / LG < 4 * NW) LG >>= 1;
    const long long out_base = offsets[v - v_lo];
    const long long slot = offsets[v - v_lo + 1] - out_base;
    if (slot == 0) continue;                           // no candidate u >= umin (the bound says so): nothing to do
    const int umin = upper ? v + 1 : 0;
    // ---- walk 1: mark every candidate ----
    walk_two_paths(rowptr, col, vs, ve, lane, LG, &s_walk, 0, MarkVisitor{bm, bm2});
    __syncthreads();
    for (int p = vs + tid; p < ve; p += LP_THREADS) {
      const int k = __ldg(col + p);
      atomicAnd(&bm[k >> 5], ~(1u << (k & 31)));
    }
    if (tid == 0) { atomicAnd(&bm[v >> 5], ~(1u << (v & 31))); s_carry = 0; s_walk = 0; }
    __syncthreads();
    // ---- rank, from block 0 (walk 3 looks up candidates below umin too) ----
    const uint32_t total = rank_blocks<LP_THREADS>(bm, bm2, blk, pre, 0, W2, s_scan, &s_carry);
    if (tid == 0) {                                    // lo = #candidates below umin
      uint32_t r = total;
      const int w0 = umin >> 5;
      if (w0 < W) {
        r = blk[w0 >> 5];
        for (uint32_t m = bm2[w0 >> 5] & ((1u << (w0 & 31)) - 1u); m; m &= m - 1) r += __popc(bm[(w0 & ~31) + __ffs(m) - 1]);
        r += __popc(bm[w0] & ((1u << (umin & 31)) - 1u));
      }
      s_lo = r;
    }
    __syncthreads();
    const uint32_t lo = s_lo;
    const bool fits = (long long)(total - lo) <= slot && (long long)total <= scratch_cap;
    if (tid == 0) counts_out[v - v_lo] = fits ? total - lo : 0xffffffffu;
    if (fits) {
      // ---- emit u >= umin into the slot (c3 zeroed), zero the c2 scratch ----
      for (int g = (umin >> 10) + tid; g < W2; g += LP_THREADS) {
        for (uint32_t m = bm2[g]; m; m &= m - 1) {
          const int w = g * 32 + __ffs(m) - 1;
          uint32_t bits = bm[w];
          uint32_t idx = blk[g] + pre[w];
          const int below = umin - (w << 5);
          if (below > 0) {
            const uint32_t mask = below >= 32 ? 0xffffffffu : ((1u << below) - 1u);
            idx += __popc(bits & mask);
            bits &= ~mask;
          }
          for (; bits; bits &= bits - 1, ++idx) {
            pad_u[out_base + (idx - lo)] = (w << 5) + __ffs(bits) - 1;
            pad_c3[out_base + (idx - lo)] = 0;
          }
        }
      }
      for (uint32_t i = tid; i < total; i += LP_THREADS) c2s[i] = 0;
      __syncthreads();
      // ---- walk 2: c2 of every candidate, tri term of the emitted ones ----
      LpScoreVisitor sv{bm, blk, pre, tri, c2s, pad_c3 + out_base, (int)lo, umin};
      walk_two_paths(rowptr, col, vs, ve, lane, LG, &s_walk, 0, sv);
      __syncthreads();
      // ---- walk 3: 32 emitted candidates per warp, handed out dynamically ----
      const int n_emit = (int)(total - lo);
      for (;;) {
        int b = 0;
        if (lane == 0) b = atomicAdd(&s_walk3, 1);
        const int e0 = __shfl_sync(FULL, b, 0) * 32;
        if (e0 >= n_emit) break;
        lp_walk3_batch(rowptr, col, bm, blk, pre, c2s, (int)lo, pad_u + out_base, pad_c2 + out_base,
                       pad_c3 + out_base, e0, min(32, n_emit - e0));
      }
      __syncthreads();
    }
    // ---- cleanup ----
    clear_blocks<LP_THREADS>(bm, bm2, 0, W2);
  }
}

// padded slot -> compact position, score from (c2, c3); work cut by compact position as in twohop_compact_kernel
__global__ void __launch_bounds__(CP_THREADS)
local_path_compact_kernel(const long long *__restrict__ pad_off, const long long *__restrict__ cmp_off, int v_lo,
                          int n_own, long long cap, const int *__restrict__ pad_u, const int *__restrict__ pad_c2,
                          const int *__restrict__ pad_c3, int *__restrict__ pair_u, int *__restrict__ pair_v,
                          float *__restrict__ score, int *__restrict__ c2_out, int *__restrict__ c3_out) {
  const long long N = cmp_off[n_own];
  if (N > cap) return;
  __shared__ int s_lo, s_hi;
  const long long ntiles = (N + CP_TILE - 1) / CP_TILE;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long base = tile * CP_TILE, end = min(base + (long long)CP_TILE, N);
    tile_owners(cmp_off, n_own, base, end, &s_lo, &s_hi);
    for (int q = 0; q < CP_PER; ++q) {
      const long long i = base + q * CP_THREADS + threadIdx.x;
      if (i >= end) break;
      int lo = s_lo;
      owner_search(cmp_off, lo, s_hi + 1, i, end);
      const long long src = pad_off[lo] + (i - cmp_off[lo]);
      const int c2 = pad_c2[src], c3 = pad_c3[src];
      pair_u[i] = pad_u[src];
      pair_v[i] = v_lo + lo;
      if (score) score[i] = local_path_score(c2, c3);
      if (c2_out) c2_out[i] = c2;
      if (c3_out) c3_out[i] = c3;
    }
  }
}

// Arbitrary pairs: a CTA takes a tile of pairs; per run of equal v it holds the N(v) bitmap, and one warp per pair walks
// N(u) (c2) and the N(j), j in N(u), as one flattened sequence (c3).  Work sum_{j in N(u)} deg j per pair: for
// evaluation sets, not for filter candidates.  Runs may come in any order; callers sort by v to make them long.
constexpr int LPP_THREADS = 512;
constexpr int LPP_TILE = 1024;

__global__ void __launch_bounds__(LPP_THREADS)
local_path_pairs_kernel(const int *__restrict__ rowptr, const int *__restrict__ col, int n, const int *__restrict__ pu,
                        const int *__restrict__ pv, long long M, float *__restrict__ score, int *__restrict__ c2_out,
                        int *__restrict__ c3_out, unsigned long long *tile_counter) {
  extern __shared__ uint32_t bitmap[];
  __shared__ long long s_tile;
  const int tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
  constexpr int NW = LPP_THREADS / 32;
  for (int w = tid; w < (n + 31) >> 5; w += LPP_THREADS) bitmap[w] = 0;
  const long long ntiles = (M + LPP_TILE - 1) / LPP_TILE;
  for (;;) {
    __syncthreads();
    if (tid == 0) s_tile = (long long)atomicAdd(tile_counter, 1ull);
    __syncthreads();
    const long long tile = s_tile;
    if (tile >= ntiles) break;
    const long long i1 = min(M, (tile + 1) * LPP_TILE);
    for (long long i = tile * LPP_TILE; i < i1;) {
      const int v = pv[i];
      long long j = i + 1;                               // end of the run (uniform: every thread scans the same pv)
      while (j < i1 && pv[j] == v) ++j;
      const int vs = __ldg(rowptr + v), ve = __ldg(rowptr + v + 1);
      for (int p = vs + tid; p < ve; p += LPP_THREADS) {
        const int k = __ldg(col + p);
        atomicOr(&bitmap[k >> 5], 1u << (k & 31));
      }
      __syncthreads();
      for (long long q = i + warp; q < j; q += NW) {
        const int u = pu[q];
        const int su = __ldg(rowptr + u), lu = __ldg(rowptr + u + 1) - su;
        int c2 = 0, c3 = 0;
        for (int base = 0; base < lu; base += 32) {
          const int p = base + lane;
          int s = 0, len = 0;
          if (p < lu) {
            const int x = __ldg(col + su + p);
            c2 += (bitmap[x >> 5] >> (x & 31)) & 1u;
            s = __ldg(rowptr + x);
            len = __ldg(rowptr + x + 1) - s;
          }
          int pin = len;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(FULL, pin, d);
            if (lane >= d) pin += t;
          }
          const int pex = pin - len;
          const int total = __shfl_sync(FULL, pin, 31);
          for (int jb = 0; jb < total; jb += 32) {
            const int pp = jb + lane;
            int sl = 0;
#pragma unroll
            for (int step = 16; step >= 1; step >>= 1) {
              const int t = __shfl_sync(FULL, pin, sl + step - 1);
              if (t <= pp) sl += step;
            }
            const int s_t = __shfl_sync(FULL, s, sl);
            const int pe_t = __shfl_sync(FULL, pex, sl);
            if (pp < total) {
              const int k = __ldg(col + s_t + (pp - pe_t));
              c3 += (bitmap[k >> 5] >> (k & 31)) & 1u;
            }
          }
        }
        c2 = __reduce_add_sync(FULL, c2);
        c3 = __reduce_add_sync(FULL, c3);
        if (lane == 0) {
          if (score) score[q] = local_path_score(c2, c3);
          if (c2_out) c2_out[q] = c2;
          if (c3_out) c3_out[q] = c3;
        }
      }
      __syncthreads();
      for (int p = vs + tid; p < ve; p += LPP_THREADS) bitmap[__ldg(col + p) >> 5] = 0;
      __syncthreads();
      i = j;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// K6 at distance 3 (eps_threehop_onepass; include/eps.h): the candidates of owner v are the ends of the 2-walks and
// 3-walks from v that are neither v nor in N(v).  A 3-walk v - k - j - u passes through a 2-walk end j, so
//   ends_3(v) = union of N(j) over j in ends_2(v) = union of N(k), k in N(v).
// One CTA per owner, enumeration only (the compaction is twohop_compact_kernel<0> without scores):
//   1. mark      ends_2 into the bitmap (walk_two_paths from every N(k), whole lists: the middle hop passes any id)
//   2. freeze    rank + list ends_2 in ascending order into a per-CTA scratch: walk 3 must not iterate the live bitmap,
//                which it fills (that would add 4-walk ends)
//   3. walk 3    N(j) for every listed j, 32 lists per warp, flattened as lp_walk3_batch (lists >= TH_LONG warp-wide),
//                atomicOr into the same bitmap; upper mode starts every N(j) at its lower bound of v + 1 and first
//                clears the ends_2 bits below v + 1
//   4. clear     N(v) and v
//   5. rank, emit ascending u into the padded slot, cleanup — as twohop_score_kernel.
// ---------------------------------------------------------------------------------------------
constexpr int TH_THREADS = 512;
constexpr int TH_LONG = 64;      // walk 3: lists at least this long are streamed warp-wide

// Walk 3 for the listed 2-walk ends e0 .. e0 + cnt - 1 (one warp): every element u >= umin of their lists is marked.
// The list was written by this CTA behind a barrier (possibly over lines an earlier owner left in L1): ld.global.cg.
__device__ __forceinline__ void threehop_walk3_batch(const int *__restrict__ rowptr, const int *__restrict__ col,
                                                     const int *ends, int e0, int cnt, int umin, MarkVisitor mv) {
  const int lane = lane_id();
  int s = 0, len = 0;
  if (lane < cnt) {
    const int j = __ldcg(ends + e0 + lane);
    s = __ldg(rowptr + j);
    const int e = __ldg(rowptr + j + 1);
    if (umin > 0) {                                      // upper-triangle mode: first position with col >= umin
      int lo = s, hi = e;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(col + mid) < umin) lo = mid + 1; else hi = mid;
      }
      s = lo;
    }
    len = e - s;
  }
  // ---- long lists: the whole warp streams one list, TS_DEPTH loads in flight per lane ----
  unsigned longmask = __ballot_sync(FULL, len >= TH_LONG);
  while (longmask) {
    const int b = __ffs(longmask) - 1;
    longmask &= longmask - 1;
    const int sb = __shfl_sync(FULL, s, b);
    const int lb = __shfl_sync(FULL, len, b);
    const int *__restrict__ lp = col + sb;
    for (int off = 0; off < lb; off += 32 * TS_DEPTH) {
      int u[TS_DEPTH];
#pragma unroll
      for (int q = 0; q < TS_DEPTH; ++q) {
        const int p = off + q * 32 + lane;
        u[q] = p < lb ? __ldg(lp + p) : -1;
      }
#pragma unroll
      for (int q = 0; q < TS_DEPTH; ++q)
        if (u[q] >= 0) mv.visit(u[q], 0);
    }
  }
  // ---- short lists: one flattened sequence ----
  const int slen = len >= TH_LONG ? 0 : len;
  int pin = slen;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int t = __shfl_up_sync(FULL, pin, d);
    if (lane >= d) pin += t;
  }
  const int pex = pin - slen;
  const int total = __shfl_sync(FULL, pin, 31);
  for (int jb = 0; jb < total; jb += 32) {
    const int p = jb + lane;
    int slot = 0;
#pragma unroll
    for (int step = 16; step >= 1; step >>= 1) {
      const int t = __shfl_sync(FULL, pin, slot + step - 1);
      if (t <= p) slot += step;
    }
    const int s_t = __shfl_sync(FULL, s, slot);
    const int pe_t = __shfl_sync(FULL, pex, slot);
    if (p < total) mv.visit(__ldg(col + s_t + (p - pe_t)), 0);
  }
}

__global__ void __launch_bounds__(TH_THREADS)
threehop_onepass_kernel(const int *__restrict__ rowptr, const int *__restrict__ col, int n, int v_lo, int v_hi,
                        const long long *__restrict__ offsets, int *__restrict__ pad_u, int *scratch,
                        long long scratch_cap, unsigned int *owner_counter, unsigned int *__restrict__ counts_out,
                        const int *__restrict__ owner_order, int n_order, int upper) {
  extern __shared__ uint32_t sm[];
  const int W = (n + 31) >> 5;
  const int W2 = (W + 31) >> 5;
  uint32_t *bm = sm;
  uint32_t *bm2 = bm + W;
  uint32_t *blk = bm2 + W2;
  uint16_t *pre = reinterpret_cast<uint16_t *>(blk + W2);
  __shared__ int s_owner, s_walk, s_walk3;
  __shared__ uint32_t s_scan[TH_THREADS / 32];
  __shared__ uint32_t s_carry;
  const int tid = threadIdx.x, lane = lane_id();
  constexpr int NW = TH_THREADS / 32;
  int *ends = scratch + (long long)blockIdx.x * scratch_cap;
  for (int w = tid; w < W + W2; w += TH_THREADS) sm[w] = 0;
  for (;;) {
    __syncthreads();
    if (tid == 0) {
      const int t = (int)atomicAdd(owner_counter, 1u);
      s_owner = (owner_order && t < n_order) ? v_lo + owner_order[t] : v_lo + t;
      s_walk = 0;
      s_walk3 = 0;
      s_carry = 0;
    }
    __syncthreads();
    const int v = s_owner;
    if (v >= v_hi) break;
    const int vs = __ldg(rowptr + v), ve = __ldg(rowptr + v + 1);
    int LG = 32;
    while (LG > 1 && (ve - vs + LG - 1) / LG < 4 * NW) LG >>= 1;
    const long long out_base = offsets[v - v_lo];
    if (offsets[v - v_lo + 1] == out_base) continue;  // no (room for) candidates (uniform): bitmap untouched
    const int umin = upper ? v + 1 : 0;
    const int g0 = umin >> 10;
    // ---- 1. mark the 2-walk ends ----
    walk_two_paths(rowptr, col, vs, ve, lane, LG, &s_walk, 0, MarkVisitor{bm, bm2});
    __syncthreads();
    // ---- 2. freeze them: ascending list in the per-CTA scratch ----
    const uint32_t n2 = rank_blocks<TH_THREADS>(bm, bm2, blk, pre, 0, W2, s_scan, &s_carry);
    if ((long long)n2 > scratch_cap) {                 // the caller's bound of the 2-walk ends is violated: poison N
      if (tid == 0) counts_out[v - v_lo] = 0xffffffffu;
      clear_blocks<TH_THREADS>(bm, bm2, 0, W2);
      continue;
    }
    for (int g = tid; g < W2; g += TH_THREADS) {
      uint32_t o = blk[g];
      for (uint32_t m = bm2[g]; m; m &= m - 1) {
        const int w = g * 32 + __ffs(m) - 1;
        for (uint32_t bits = bm[w]; bits; bits &= bits - 1) ends[o++] = (w << 5) + __ffs(bits) - 1;
      }
    }
    __syncthreads();
    if (upper) {                                       // keep only marks >= umin: blocks below g0, then words below umin
      clear_blocks<TH_THREADS>(bm, bm2, 0, g0);
      const int w0 = umin >> 5;
      for (int w = g0 * 32 + tid; w <= w0 && w < W; w += TH_THREADS)
        bm[w] &= w < w0 ? 0u : ~((1u << (umin & 31)) - 1u);
    }
    __syncthreads();
    // ---- 3. walk 3: N(j) of every 2-walk end j, 32 lists per warp, handed out dynamically ----
    for (;;) {
      int b = 0;
      if (lane == 0) b = atomicAdd(&s_walk3, 1);
      const int e0 = __shfl_sync(FULL, b, 0) * 32;
      if (e0 >= (int)n2) break;
      threehop_walk3_batch(rowptr, col, ends, e0, min(32, (int)n2 - e0), umin, MarkVisitor{bm, bm2});
    }
    __syncthreads();
    // ---- 4. clear known edges and the diagonal ----
    for (int p = vs + tid; p < ve; p += TH_THREADS) {
      const int k = __ldg(col + p);
      if (k >= umin) atomicAnd(&bm[k >> 5], ~(1u << (k & 31)));
    }
    if (tid == 0) {
      if (v >= umin) atomicAnd(&bm[v >> 5], ~(1u << (v & 31)));
      s_carry = 0;
    }
    __syncthreads();
    // ---- 5. rank, emit ascending u, cleanup ----
    const uint32_t total = rank_blocks<TH_THREADS>(bm, bm2, blk, pre, g0, W2, s_scan, &s_carry);
    const bool fits = (long long)total <= offsets[v - v_lo + 1] - out_base;
    if (tid == 0) counts_out[v - v_lo] = fits ? total : 0xffffffffu;
    if (fits) {
      for (int g = g0 + tid; g < W2; g += TH_THREADS) {
        long long o = out_base + blk[g];
        for (uint32_t m = bm2[g]; m; m &= m - 1) {
          const int w = g * 32 + __ffs(m) - 1;
          for (uint32_t bits = bm[w]; bits; bits &= bits - 1) pad_u[o++] = (w << 5) + __ffs(bits) - 1;
        }
      }
    }
    __syncthreads();
    clear_blocks<TH_THREADS>(bm, bm2, g0, W2);
  }
}

}  // namespace eps

extern "C" int eps_score_kinds(void) {
  return (1 << eps::score_kind(EPS_SCORE_JACCARD)) | (1 << eps::score_kind(EPS_SCORE_SORENSEN)) |
         (1 << eps::score_kind(EPS_SCORE_SALTON)) | (1 << eps::score_kind(EPS_SCORE_HUB_PROMOTED)) |
         (1 << eps::score_kind(EPS_SCORE_HUB_DEPRESSED)) | (1 << eps::score_kind(EPS_SCORE_LHN)) |
         (1 << eps::score_kind(EPS_SCORE_PREF_ATTACH));
}

// ---------------------------------------------------------------------------------------------
// Host plan of the one-pass entry points (eps_twohop_onepass, eps_local_path_onepass).  Workspace:
//   ticket (256 B) | 64 work buckets (256 B) | per-owner counts | owner order | the entry point's padded slots ...
// ---------------------------------------------------------------------------------------------
static inline size_t up256(size_t x) { return (x + 255) & ~(size_t)255; }
static inline size_t onepass_header_bytes(size_t n_own) { return 512 + 2 * up256(n_own * 4); }

namespace eps {

struct OnepassPlan {
  size_t smem;                  // one owner's bitmap and rank tables
  unsigned int *ticket, *buckets, *counts;
  int *order;
  uint8_t *slots;               // the padded slots behind the header
  int cgrid;                    // grid of the compaction pass
};

// The owner bitmap's shared memory (<= 200 KB) and the workspace header; zeroes the ticket, buckets and counts.
static int onepass_begin(const char *what, int n, int n_own, void *workspace, cudaStream_t stream, OnepassPlan &p) {
  const int W = (n + 31) / 32, W2 = (W + 31) / 32;
  p.smem = (size_t)(W + 2 * W2) * 4 + (size_t)W * 2 + 16;
  if (p.smem > 200 * 1024) {
    set_error("%s: n=%d needs %zu bytes of shared memory (> 200 KB)", what, n, p.smem);
    return EPS_ERR_UNSUPPORTED;
  }
  uint8_t *ws = (uint8_t *)workspace;
  p.ticket = (unsigned int *)ws;
  p.buckets = (unsigned int *)(ws + 256);
  p.counts = (unsigned int *)(ws + 512);
  p.order = (int *)(ws + 512 + up256((size_t)n_own * 4));
  p.slots = ws + onepass_header_bytes(n_own);
  EPS_CUDA(cudaMemsetAsync(ws, 0, 512 + up256((size_t)n_own * 4), stream));   // ticket + buckets + counts
  return EPS_OK;
}

// Heaviest-first owner order, the owner kernel on as many CTAs as fit (at most max_ctas), the scan of the real counts
// into offsets_out; sets the compaction grid.
template <typename... P, typename... A>
static int onepass_run(OnepassPlan &p, void (*kern)(P...), int threads, long long max_ctas, int n_own,
                       const int64_t *bound_offsets, int64_t cap, int64_t *offsets_out, int sms, cudaStream_t stream,
                       A... args) {
  EPS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  int occ = 0;
  EPS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, p.smem));
  if (occ < 1) occ = 1;
  const int grid = (int)std::min<long long>(std::min<long long>((long long)n_own, (long long)sms * occ), max_ctas);
  {  // heaviest-first hand-out: counting sort of the owners by the power of two of their slot size (the bound)
    const int ogrid = std::min((n_own + 255) / 256, sms * 8);
    owner_bucket_kernel<0><<<ogrid, 256, 0, stream>>>((const long long *)bound_offsets, n_own, p.buckets, p.order);
    owner_bucket_kernel<1><<<1, 64, 0, stream>>>((const long long *)bound_offsets, n_own, p.buckets, p.order);
    owner_bucket_kernel<2><<<ogrid, 256, 0, stream>>>((const long long *)bound_offsets, n_own, p.buckets, p.order);
    EPS_LAUNCH_CHECK();
  }
  kern<<<grid, threads, p.smem, stream>>>(args...);
  EPS_LAUNCH_CHECK();
  owner_scan_kernel<<<1, 1024, 0, stream>>>(p.counts, n_own, (long long *)offsets_out);
  EPS_LAUNCH_CHECK();
  p.cgrid = (int)std::min<long long>((cap + CP_TILE - 1) / CP_TILE, (long long)sms * 8);
  return EPS_OK;
}

using ScoreKernel = void (*)(const int *, const int *, const float *, const float *, int, int, int, const long long *,
                             int *, int, int, unsigned long long *, int *, unsigned int *, unsigned int *, const int *);
// index [HAS_W][WANT_CN][HAS_VAL]
static const ScoreKernel kScoreKernels[2][2][2] = {
    {{twohop_score_kernel<false, false, false>, twohop_score_kernel<false, false, true>},
     {twohop_score_kernel<false, true, false>, twohop_score_kernel<false, true, true>}},
    {{twohop_score_kernel<true, false, false>, twohop_score_kernel<true, false, true>},
     {twohop_score_kernel<true, true, false>, twohop_score_kernel<true, true, true>}}};

}  // namespace eps

extern "C" size_t eps_twohop_onepass_workspace_bytes(int64_t cap, int32_t n_owners) {
  const size_t c = (size_t)(cap > 0 ? cap : 0), o = (size_t)(n_owners > 0 ? n_owners : 0);
  // header | padded u | padded CN counts | padded fixed-point sums
  return onepass_header_bytes(o) + up256(c * 4) + up256(c * 4) + up256(c * 8);
}

extern "C" int eps_twohop_onepass(const int32_t *rowptr, const int32_t *col, const float *val,
                                  const float *wtable, int32_t n, int32_t v_lo, int32_t v_hi, const int64_t *bound_offsets,
                                  int64_t cap, int flags, int32_t *pair_u, int32_t *pair_v, float *score,
                                  int32_t *count, int64_t *offsets_out, void *workspace,
                                  size_t workspace_bytes, void *stream_) {
  using namespace eps;
  cudaStream_t stream = (cudaStream_t)stream_;
  EPS_CHECK_ARG(rowptr && col && bound_offsets && offsets_out, "null graph, bound_offsets or offsets_out pointer");
  EPS_CHECK_ARG(n > 0 && v_lo >= 0 && v_hi <= n && v_lo < v_hi && cap >= 0, "bad owner range or cap");
  EPS_CHECK_ARG(cap == 0 || (pair_u && pair_v), "missing pair output pointer");
  EPS_CHECK_ARG(!(wtable && !score), "wtable given but no score output");
  EPS_CHECK_ARG(!(val && !score), "edge values given but no score output");
  EPS_CHECK_ARG(!(flags & ~(EPS_CN_SIGMOID | EPS_TWOHOP_UPPER | EPS_SCORE_KIND_MASK)), "unknown flag bits");
  const int kind = score_kind(flags);
  EPS_CHECK_ARG(!kind || (!wtable && !val && !(flags & EPS_CN_SIGMOID)),
                "a similarity kind (EPS_SCORE_*) needs wtable == NULL, val == NULL and no EPS_CN_SIGMOID");
  const int sms = sm_count();
  if (sms <= 0) { set_error("eps_twohop_onepass: no CUDA device"); return EPS_ERR_CUDA; }
  const int n_own = v_hi - v_lo;
  if (!workspace || workspace_bytes < eps_twohop_onepass_workspace_bytes(cap, n_own)) {
    set_error("eps_twohop_onepass: workspace too small");
    return EPS_ERR_WORKSPACE;
  }
  OnepassPlan p;
  if (const int st = onepass_begin("eps_twohop_onepass", n, n_own, workspace, stream, p)) return st;
  int *pad_u = (int *)p.slots;
  int *pad_cn = (int *)((uint8_t *)pad_u + up256((size_t)cap * 4));
  unsigned long long *pad_acc = (unsigned long long *)((uint8_t *)pad_cn + up256((size_t)cap * 4));
  const bool want_score = score != nullptr || count != nullptr;
  unsigned long long *acc = nullptr;
  int *cn = nullptr;
  if (wtable || val) {
    acc = pad_acc;
    EPS_CUDA(cudaMemsetAsync(acc, 0, (size_t)cap * 8, stream));
    if (count) cn = pad_cn;
  } else if (want_score) {
    cn = pad_cn;
  }
  if (cn) EPS_CUDA(cudaMemsetAsync(cn, 0, (size_t)cap * 4, stream));
  if (const int st = onepass_run(p, kScoreKernels[wtable != nullptr][cn != nullptr][val != nullptr], TS_THREADS, n_own,
                                 n_own, bound_offsets, cap, offsets_out, sms, stream, rowptr, col, val, wtable, n, v_lo,
                                 v_hi, (const long long *)bound_offsets, pad_u, n_own, (flags & EPS_TWOHOP_UPPER) ? 1 : 0,
                                 acc, cn, p.ticket, p.counts, p.order))
    return st;
  if (cap > 0) {
    kCompactKinds[kind]<<<p.cgrid, CP_THREADS, 0, stream>>>(rowptr, (const long long *)bound_offsets,
                                                           (const long long *)offsets_out, v_lo, n_own, (long long)cap,
                                                           pad_u, acc, cn, flags, pair_u, pair_v, score, count);
    EPS_LAUNCH_CHECK();
  }
  return EPS_OK;
}

// ---------------------------------------------------------------------------------------------
// Local Path index entry points
// ---------------------------------------------------------------------------------------------
extern "C" size_t eps_local_path_onepass_workspace_bytes(int64_t cap, int32_t n_owners, int64_t max_count,
                                                         int32_t ctas) {
  const size_t c = (size_t)(cap > 0 ? cap : 0), o = (size_t)(n_owners > 0 ? n_owners : 0);
  const size_t s = (size_t)(max_count > 0 ? max_count : 0) * (size_t)(ctas > 0 ? ctas : 0);
  // header | padded u | padded c2 | padded c3 | per-CTA c2 scratch
  return onepass_header_bytes(o) + 3 * up256(c * 4) + up256(s * 4);
}

extern "C" int eps_local_path_onepass(const int32_t *rowptr, const int32_t *col, const int32_t *tri, int32_t n,
                                      int32_t v_lo, int32_t v_hi, const int64_t *bound_offsets, int64_t cap,
                                      int64_t max_count, int32_t ctas, int flags, int32_t *pair_u, int32_t *pair_v,
                                      float *score, int32_t *c2, int32_t *c3, int64_t *offsets_out, void *workspace,
                                      size_t workspace_bytes, void *stream_) {
  using namespace eps;
  cudaStream_t stream = (cudaStream_t)stream_;
  EPS_CHECK_ARG(rowptr && col && tri && bound_offsets && offsets_out,
                "null graph, tri, bound_offsets or offsets_out pointer");
  EPS_CHECK_ARG(n > 0 && v_lo >= 0 && v_hi <= n && v_lo < v_hi && cap >= 0 && cap < (1ll << 31),
                "bad owner range or cap");
  EPS_CHECK_ARG(max_count >= 0 && max_count < (1ll << 31) && ctas >= 1, "bad max_count or ctas");
  EPS_CHECK_ARG(cap == 0 || (pair_u && pair_v), "missing pair output pointer");
  EPS_CHECK_ARG(!(flags & ~EPS_TWOHOP_UPPER), "unknown flag bits");
  const int n_own = v_hi - v_lo;
  if (!workspace || workspace_bytes < eps_local_path_onepass_workspace_bytes(cap, n_own, max_count, ctas)) {
    set_error("eps_local_path_onepass: workspace too small");
    return EPS_ERR_WORKSPACE;
  }
  const int sms = sm_count();
  if (sms <= 0) { set_error("eps_local_path_onepass: no CUDA device"); return EPS_ERR_CUDA; }
  OnepassPlan p;
  if (const int st = onepass_begin("eps_local_path_onepass", n, n_own, workspace, stream, p)) return st;
  int *pad_u = (int *)p.slots;
  int *pad_c2 = (int *)((uint8_t *)pad_u + up256((size_t)cap * 4));
  int *pad_c3 = (int *)((uint8_t *)pad_c2 + up256((size_t)cap * 4));
  int *scratch = (int *)((uint8_t *)pad_c3 + up256((size_t)cap * 4));
  if (const int st = onepass_run(p, local_path_onepass_kernel, LP_THREADS, ctas, n_own, bound_offsets, cap, offsets_out,
                                 sms, stream, rowptr, col, tri, n, v_lo, v_hi, (const long long *)bound_offsets, pad_u,
                                 pad_c2, pad_c3, scratch, (long long)max_count, p.ticket, p.counts, p.order, n_own,
                                 (flags & EPS_TWOHOP_UPPER) ? 1 : 0))
    return st;
  if (cap > 0) {
    local_path_compact_kernel<<<p.cgrid, CP_THREADS, 0, stream>>>((const long long *)bound_offsets,
                                                                (const long long *)offsets_out, v_lo, n_own,
                                                                (long long)cap, pad_u, pad_c2, pad_c3, pair_u, pair_v,
                                                                score, c2, c3);
    EPS_LAUNCH_CHECK();
  }
  return EPS_OK;
}

extern "C" size_t eps_local_path_pairs_workspace_bytes(void) { return 256; }

extern "C" int eps_local_path_pairs(const int32_t *rowptr, const int32_t *col, int32_t n, const int32_t *pair_u,
                                    const int32_t *pair_v, int64_t M, int flags, float *score, int32_t *c2,
                                    int32_t *c3, void *workspace, size_t workspace_bytes, void *stream_) {
  using namespace eps;
  cudaStream_t stream = (cudaStream_t)stream_;
  EPS_CHECK_ARG(n > 0 && M >= 0, "bad n or M");
  EPS_CHECK_ARG(flags == 0, "unknown flag bits");
  if (M == 0) return EPS_OK;
  EPS_CHECK_ARG(rowptr && col && pair_u && pair_v, "null graph or pair pointer");
  EPS_CHECK_ARG(score || c2 || c3, "score, c2 and c3 all NULL");
  if (!workspace || workspace_bytes < eps_local_path_pairs_workspace_bytes()) {
    set_error("eps_local_path_pairs: workspace too small");
    return EPS_ERR_WORKSPACE;
  }
  const size_t bitmap_bytes = (size_t)((n + 31) / 32) * 4;
  if (bitmap_bytes > 200 * 1024) {
    set_error("eps_local_path_pairs: n=%d needs %zu bytes of shared memory (> 200 KB)", n, bitmap_bytes);
    return EPS_ERR_UNSUPPORTED;
  }
  const int sms = sm_count();
  if (sms <= 0) { set_error("eps_local_path_pairs: no CUDA device"); return EPS_ERR_CUDA; }
  EPS_CUDA(cudaMemsetAsync(workspace, 0, 8, stream));
  EPS_CUDA(cudaFuncSetAttribute(local_path_pairs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)bitmap_bytes));
  int occ = 0;
  EPS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, local_path_pairs_kernel, LPP_THREADS, bitmap_bytes));
  if (occ < 1) occ = 1;
  const long long ntiles = (M + LPP_TILE - 1) / LPP_TILE;
  const int grid = (int)std::min<long long>(ntiles, (long long)sms * occ);
  local_path_pairs_kernel<<<grid, LPP_THREADS, bitmap_bytes, stream>>>(rowptr, col, n, pair_u, pair_v, (long long)M,
                                                                     score, c2, c3, (unsigned long long *)workspace);
  EPS_LAUNCH_CHECK();
  return EPS_OK;
}

// ---------------------------------------------------------------------------------------------
// Distance-3 enumeration entry point
// ---------------------------------------------------------------------------------------------
extern "C" size_t eps_threehop_onepass_workspace_bytes(int64_t cap, int32_t n_owners, int64_t max_ends, int32_t ctas) {
  const size_t c = (size_t)(cap > 0 ? cap : 0), o = (size_t)(n_owners > 0 ? n_owners : 0);
  const size_t s = (size_t)(max_ends > 0 ? max_ends : 0) * (size_t)(ctas > 0 ? ctas : 0);
  // header | padded u | per-CTA list of the 2-walk ends
  return onepass_header_bytes(o) + up256(c * 4) + up256(s * 4);
}

extern "C" int eps_threehop_onepass(const int32_t *rowptr, const int32_t *col, int32_t n, int32_t v_lo, int32_t v_hi,
                                    const int64_t *bound_offsets, int64_t cap, int64_t max_ends, int32_t ctas, int flags,
                                    int32_t *pair_u, int32_t *pair_v, int64_t *offsets_out, void *workspace,
                                    size_t workspace_bytes, void *stream_) {
  using namespace eps;
  cudaStream_t stream = (cudaStream_t)stream_;
  EPS_CHECK_ARG(rowptr && col && bound_offsets && offsets_out, "null graph, bound_offsets or offsets_out pointer");
  EPS_CHECK_ARG(n > 0 && v_lo >= 0 && v_hi <= n && v_lo < v_hi && cap >= 0 && cap < (1ll << 31),
                "bad owner range or cap");
  EPS_CHECK_ARG(max_ends >= 0 && max_ends < (1ll << 31) && ctas >= 1, "bad max_ends or ctas");
  EPS_CHECK_ARG(cap == 0 || (pair_u && pair_v), "missing pair output pointer");
  EPS_CHECK_ARG(!(flags & ~EPS_TWOHOP_UPPER), "unknown flag bits");
  const int n_own = v_hi - v_lo;
  if (!workspace || workspace_bytes < eps_threehop_onepass_workspace_bytes(cap, n_own, max_ends, ctas)) {
    set_error("eps_threehop_onepass: workspace too small");
    return EPS_ERR_WORKSPACE;
  }
  const int sms = sm_count();
  if (sms <= 0) { set_error("eps_threehop_onepass: no CUDA device"); return EPS_ERR_CUDA; }
  OnepassPlan p;
  if (const int st = onepass_begin("eps_threehop_onepass", n, n_own, workspace, stream, p)) return st;
  int *pad_u = (int *)p.slots;
  int *scratch = (int *)((uint8_t *)pad_u + up256((size_t)cap * 4));
  if (const int st = onepass_run(p, threehop_onepass_kernel, TH_THREADS, ctas, n_own, bound_offsets, cap, offsets_out,
                                 sms, stream, rowptr, col, n, v_lo, v_hi, (const long long *)bound_offsets, pad_u,
                                 scratch, (long long)max_ends, p.ticket, p.counts, p.order, n_own,
                                 (flags & EPS_TWOHOP_UPPER) ? 1 : 0))
    return st;
  if (cap > 0) {
    twohop_compact_kernel<0><<<p.cgrid, CP_THREADS, 0, stream>>>(rowptr, (const long long *)bound_offsets,
                                                                (const long long *)offsets_out, v_lo, n_own,
                                                                (long long)cap, pad_u, nullptr, nullptr, 0, pair_u,
                                                                pair_v, nullptr, nullptr);
    EPS_LAUNCH_CHECK();
  }
  return EPS_OK;
}
