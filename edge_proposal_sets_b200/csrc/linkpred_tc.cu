// K2 (tensor-core arm) — fused gather + Hadamard + LinkPredictor MLP on tcgen05 / TMEM.
//
// Replaces /root/reference/models.py:506 (two row gathers) + models.py:478-485 (LinkPredictor), i.e.
// index_select x2, mul, (cuBLAS SGEMM + bias + relu) x (L-1), GEMV, sigmoid — 2L+3 launches and 2*B*H*4 bytes of
// materialised gathers per batch in the reference.  Operands are IEEE fp16 under a device-computed power-of-two
// scale (tc_common.cuh), accumulation / output layer / sigmoid are fp32.
// A cluster of two CTAs (tcgen05 cta_group::2) keeps its halves of ALL hidden-layer weights resident
// in shared memory (with H = 256 one layer's fp16 weights are 128 KB: the pair splits the N dimension of the
// B operand, 64 KB per SM and layer) and runs warp-specialised roles per CTA, connected by mbarriers:
//
//   ids warp             (u, v) of a tile's 128 rows -> shared memory one tile ahead, plus the h[v] ROWS of the tile's
//                        owners (the list is grouped by v: one owner per tile, now and then two) staged in shared memory;
//   loaders (4 warps)    cp.async (LDGSTS) of the h[u] pieces of every 128 x 32 K-chunk straight into a ring of 8 KB
//                        stages (K-major SWIZZLE_64B), completion counted on the stage's mbarrier: the whole ring
//                        (9 stages at H = 256, L = 3) is in flight ahead of the tensor pipe and nobody waits for data;
//   producers (4 warps)  multiply a landed chunk in place by h[v] (HMUL2, operands from shared memory only),
//                        fence.proxy.async, hand the stage to the MMA issuer;
//   MMA issuer (1 lane,  waits for a ring stage from BOTH CTAs, issues M=256 x N=H x K=16 UMMAs
//   leader CTA only)     into one of two TMEM accumulator slots, releases stages / publishes accumulators with
//                        multicast tcgen05.commit; layers after the first read their A operand from TENSOR MEMORY;
//   epilogue (4 warps)   thread-per-row: tcgen05.ld, ReLU, then either round to fp16 and tcgen05.st the packed chunk
//                        back into the accumulator slot IN PLACE — it becomes the next layer's A operand, published
//                        per 32-column chunk so the next layer's MMAs trail the conversion, and the activations never
//                        touch shared memory — or the fused H -> 1 output layer + sigmoid.
//
// The two accumulator slots let the tensor pipe start the next GEMM (next layer, or next tile's first layer) while
// the epilogue drains the previous one; the ring decouples the HBM/L2 gather from both.  Short pair lists (no fp16
// table) gather fp32 rows through registers instead (two producer groups, no loaders).
// How the design got here, with the measurements behind every step: profiles/round2_d_k2_timeline.md.
#include <cooperative_groups.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "tc_common.cuh"

namespace eps {

namespace cg = cooperative_groups;

constexpr int P_MAX_RING = 10;                                     // first-layer ring stages (8 KB each), chosen at launch
constexpr int P_VROWS = 4;                                         // distinct owners of a 128-row tile whose h[v] row is staged
constexpr int P_MAX_CHUNKS = 8;                                    // 32-column K-chunks per layer at H = 256
constexpr int P_GROUP_WARPS = 4;                                   // warps per producer group
// Warp roles: 4 epilogue warps (one per TMEM lane quarter), then the MMA warp, the pair-id warp, NL loader warps
// (fp16-table path) and NG producer groups of four warps each.
//   fp16 table: NL = 4 loaders + NG = 1 group multiplying in place.  4 or 8 loaders with 1 or 2 groups all ran within
//               3 % (profiles/round2_d_k2_timeline.md, step 11); this is the shape with the fewest warps.
//   fp32 source (short lists): NL = 0, NG = 2 groups that load through registers.
constexpr int p_groups(bool hb) { return hb ? 1 : 2; }
constexpr int p_loaders(bool hb) { return hb ? 4 : 0; }
// one CTA per SM: the whole register file is there to be used
// (16384 registers per SM sub-partition, warps dealt round-robin: 14 warps -> 4 on one -> 128)
constexpr int P_EPI_WARPS = 4;                                     // one per TMEM lane quarter
constexpr int p_threads(bool hb) { return (P_EPI_WARPS + 2 + p_loaders(hb) + p_groups(hb) * P_GROUP_WARPS) * 32; }
constexpr int p_maxreg(bool hb) { return (16384 / (((p_threads(hb) / 32) + 3) / 4) / 32) / 8 * 8; }
constexpr int P_CHUNK_K = 32;
constexpr int P_STAGE_BYTES = TC_BM * P_CHUNK_K * 2;               // 8 KB

__device__ __forceinline__ uint64_t umma_smem_desc_sw64(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512u >> 4) << 32;                // 8 rows x 64 B
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;                          // SWIZZLE_64B
  return d;
}
// 16-wide K tiles (one UMMA K step, 32-byte rows) in K-major SWIZZLE_32B: 8-row groups 256 B apart,
// 16-byte chunk index ^= bit 7 of the byte offset = (r >> 2) & 1
__device__ __forceinline__ uint64_t umma_smem_desc_sw32(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(256u >> 4) << 32;                // 8 rows x 32 B
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)6 << 61;                          // SWIZZLE_32B
  return d;
}
__device__ __forceinline__ uint32_t sw32_chunk_off(int r, int chunk) {
  return (uint32_t)r * 32u + (uint32_t)((chunk ^ ((r >> 2) & 1)) << 4);
}
// tcgen05.ld of 16 accumulator columns WITHOUT the wait, and a wait that names the destination
// registers so no use of them can be scheduled above it: the epilogue keeps the next load in
// flight while it converts the current one.
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t *r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait16(uint32_t *r) {
  asm volatile(
      "tcgen05.wait::ld.sync.aligned;\n"
      : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
        "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
      :: "memory");
}
__device__ __forceinline__ uint32_t sw64_chunk_off(int r, int sub) {
  return (uint32_t)r * 64u + (uint32_t)((sub ^ ((r >> 1) & 3)) << 4);
}
__device__ __forceinline__ void umma_f16_ss_2cta_p(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                                    uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}\n"
      :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
// A operand from TENSOR MEMORY (lane = row, one 32-bit column = two consecutive K elements), B from shared memory
__device__ __forceinline__ void umma_f16_ts_2cta_p(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc,
                                                    uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}\n"
      :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t *r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n"
      :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
         "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void umma_commit_mc(uint32_t mbar_saddr) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      :: "r"(mbar_saddr), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void mbar_arrive_on_cta(uint32_t local_saddr, uint32_t target_cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_saddr), "r"(target_cta));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" :: "r"(r) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t saddr, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "DONE:\n\t}\n"
      :: "r"(saddr), "r"(parity) : "memory");
}

// Optional timeline trace of cluster 0 (build with -DEPS_TC3_TRACE; tools/tc3_trace.py reads the dump):
// one record per pipeline event = tag | a | b | clock64 of the leader CTA's SM.
#ifdef EPS_TC3_TRACE
// fire-and-forget stores into a per-role region (MMA issuer 0, epilogue 1, producer group g 2+g); no atomics
constexpr unsigned TR_REGION = 1u << 15;
__device__ unsigned long long g_trace[8 * TR_REGION];
#define TR_DECL(role) unsigned tr_n_ = 0; const unsigned tr_base_ = (unsigned)(role) * TR_REGION
#define TR(tag, a, b)                                                                                  \
  do {                                                                                                 \
    if (cluster_id == 0 && cta_rank == 0 && tr_n_ < TR_REGION)                                         \
      g_trace[tr_base_ + tr_n_++] = ((unsigned long long)(tag) << 56) | ((unsigned long long)((a) & 0xff) << 48) | \
                      ((unsigned long long)((b) & 0xff) << 40) | ((unsigned long long)clock64() & 0xffffffffffull); \
  } while (0)
#else
#define TR_DECL(role) do { } while (0)
#define TR(tag, a, b) do { } while (0)
#endif

// one non-blocking look at a barrier phase (the blocking form may park the thread for a while)
__device__ __forceinline__ uint32_t mbar_test(uint32_t saddr, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t}\n"
      : "=r"(ok) : "r"(saddr), "r"(parity) : "memory");
  return ok;
}

struct PipeBarriers {
  uint64_t full[P_MAX_RING];   // producers (both CTAs) -> MMA issuer       (waited in the leader)
  uint64_t empty[P_MAX_RING];  // MMA commit -> whoever refills the stage    (multicast, both CTAs)
  uint64_t landed[P_MAX_RING]; // loader warps' copies (cp.async completion) -> producers   (CTA-local; fp16-table path)
  uint64_t acc_full[2];        // MMA commit -> epilogue                     (multicast, both CTAs)
  uint64_t acc_free[2];        // epilogue (both CTAs) -> MMA issuer         (waited in the leader)
  uint64_t a2_full[P_MAX_CHUNKS];  // epilogue (both CTAs) -> MMA issuer: 32-column chunk c of the activations is in TMEM
  uint64_t ids_full[2];        // ids warp -> producers                      (CTA-local)
  uint64_t ids_empty[2];       // producers -> ids warp                      (CTA-local)
  uint64_t wload;              // TMA bulk copies of the resident weights -> everyone (once per kernel)
  uint32_t tmem_base_slot;
};

__device__ __forceinline__ uint32_t cvt_relu_f16x2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));   // max(x, 0) then RN to fp16
  return d;
}
__device__ __forceinline__ float2 fma_f32x2(float2 a, float2 b, float2 c) {
  unsigned long long pa, pb, pc, pr;
  asm("mov.b64 %0, {%1, %2};" : "=l"(pa) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(pb) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(pc) : "f"(c.x), "f"(c.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(pr) : "l"(pa), "l"(pb), "l"(pc));
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(pr));
  return r;
}
template <int H, bool HB /* h is the fp16 table (else fp32) */>
__global__ void __cluster_dims__(2, 1, 1) __maxnreg__(p_maxreg(HB))
linkpred_tc3_kernel(const void *__restrict__ h, const int *__restrict__ pu, const int *__restrict__ pv,
                    long long M, const MlpParams prm, int L, int apply_sigmoid,
                    const uint8_t *__restrict__ wimg, float *__restrict__ score, int ring,
                    const TcScale *__restrict__ scale) {
  static_assert(H % 64 == 0 && H >= 64 && H <= 256, "H in {64,128,192,256}");
  constexpr int NG = p_groups(HB), NL = p_loaders(HB);       // producer groups, loader warps
  constexpr int HH = H / 2;
  constexpr int WH_BYTES = HH * H * 2;
  constexpr int NCHUNK = H / P_CHUNK_K;                       // 32-column K-chunks per layer (8 KB of A operand each)
  constexpr int P_IDS_WARP = P_EPI_WARPS + 1, P_FIRST_LOAD_WARP = P_EPI_WARPS + 2, P_FIRST_PROD_WARP = P_FIRST_LOAD_WARP + NL;
  constexpr int P_THREADS = p_threads(HB);
  constexpr int P_PROD_WARPS = NG * P_GROUP_WARPS;
  constexpr uint32_t TMEM_COLS = 2 * H <= 128 ? 128 : (2 * H <= 256 ? 256 : 512);
  constexpr uint32_t IDESC = umma_idesc_f16(2 * TC_BM, H);
  // ALL shared memory is dynamic and laid out by hand (no alignment pad: the window itself is 1 KB
  // aligned — checked below — and every swizzled region starts at a multiple of 1 KB).  With H = 256
  // and two hidden layers the resident weights take 128 KB; the rest is the ring of the first layer's
  // A operand: `ring` stages (as many as fit, 10 at H = 256) of one 8 KB K-chunk (128 rows x 32 K, SWIZZLE_64B).
  // The later layers take their A operand from TENSOR memory (see the epilogue), not from here.
  extern __shared__ __align__(1024) uint8_t smem[];
  const int nhidden = L - 1;
  uint8_t *sW = smem;                                                   // [nhidden][WH_BYTES]
  uint8_t *sRing = sW + (size_t)nhidden * WH_BYTES;                     // [ring][8 KB]
  uint8_t *sOnes = sRing + (size_t)ring * P_STAGE_BYTES;                // [128][16] fp16: A of the bias K-step
  uint8_t *sBiasB = sOnes + TC_BM * 32;                                 // [nhidden][HH][16] fp16: B of the bias K-step
  float *sWlast = reinterpret_cast<float *>(sBiasB + (size_t)nhidden * HH * 32);   // [H]
  int2 *sIds = reinterpret_cast<int2 *>(sWlast + H);                    // [2][128] (u, v) of this CTA's rows
  int *sKi = reinterpret_cast<int *>(sIds + 2 * TC_BM);                 // [2][128] index of the row's v in sV (-1: not cached)
  uint8_t *sV = reinterpret_cast<uint8_t *>(sKi + 2 * TC_BM);           // [2][P_VROWS][H] fp16: h[v] rows of the tile's owners
  int *sVid = reinterpret_cast<int *>(sV + (HB ? 2 * P_VROWS * H * 2 : 0));   // [P_VROWS] scratch of the ids warp
  PipeBarriers &bars = *reinterpret_cast<PipeBarriers *>(sVid + 8);
  cg::cluster_group cluster = cg::this_cluster();
  const uint32_t cta_rank = cluster.block_rank();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  const float hscale = scale->hscale, S = scale->S, invS = scale->invS;

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(smem_u32(&bars.tmem_base_slot)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
    for (int i = 0; i < P_MAX_RING; ++i) {
      mbar_init(smem_u32(&bars.full[i]), 2 * P_GROUP_WARPS);
      mbar_init(smem_u32(&bars.empty[i]), 1);
      mbar_init(smem_u32(&bars.landed[i]), NL > 0 ? NL * 32 : 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&bars.acc_full[i]), 1);
      mbar_init(smem_u32(&bars.acc_free[i]), 2 * P_EPI_WARPS);
    }
    for (int i = 0; i < P_MAX_CHUNKS; ++i) mbar_init(smem_u32(&bars.a2_full[i]), 2 * P_EPI_WARPS);
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&bars.ids_full[i]), 1);
      mbar_init(smem_u32(&bars.ids_empty[i]), P_PROD_WARPS + NL);
    }
    mbar_init(smem_u32(&bars.wload), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    // The resident weights: this CTA's half of every hidden layer's pre-swizzled image (64 KB per layer at H = 256) comes
    // in with one TMA bulk copy per layer (cp.async.bulk, SASS UBLKCP) straight from the async proxy the MMA reads
    // with — no registers, no generic-proxy stores to fence; everybody waits for the byte count below.
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                 :: "r"(smem_u32(&bars.wload)), "r"((uint32_t)(nhidden * WH_BYTES)) : "memory");
    for (int l = 0; l < nhidden; ++l)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   :: "r"(smem_u32(sW + (size_t)l * WH_BYTES)),
                      "l"(wimg + (size_t)l * H * H * 2 + (size_t)cta_rank * WH_BYTES), "r"((uint32_t)WH_BYTES),
                      "r"(smem_u32(&bars.wload)) : "memory");
  }
  // Biases ride in the MMA: one extra K = 16 step per hidden layer with A = [1 1 1 0 ...] for every
  // row and B[n] = [hi mid lo 0 ...], S times the bias of output feature n split into three fp16 terms
  // (hi + mid + lo reproduces the fp32 value exactly: 3 x 11 significand bits).  The epilogue then never touches shared
  // memory for a bias, and the accumulator is initialised by this step instead of a zeroing MMA flag.
  for (int i = tid; i < TC_BM; i += P_THREADS) {
    const uint32_t one2 = 0x3C003C00u;                               // fp16 (1, 1)
    *reinterpret_cast<uint4 *>(sOnes + sw32_chunk_off(i, 0)) = make_uint4(one2, 0x00003C00u, 0u, 0u);
    *reinterpret_cast<uint4 *>(sOnes + sw32_chunk_off(i, 1)) = make_uint4(0u, 0u, 0u, 0u);
  }
  for (int i = tid; i < nhidden * HH; i += P_THREADS) {
    const int l = i / HH, r = i - l * HH;
    const float b = __ldg(prm.b[l] + cta_rank * HH + r) * S;     // hidden activations are carried times S
    const __half hi = __float2half_rn(b);
    const float r1 = b - __half2float(hi);
    const __half mid = __float2half_rn(r1);
    const __half lo = __float2half_rn(r1 - __half2float(mid));
    const uint32_t w0 = (uint32_t)__half_as_ushort(hi) | ((uint32_t)__half_as_ushort(mid) << 16);
    uint8_t *t = sBiasB + (size_t)l * HH * 32;
    *reinterpret_cast<uint4 *>(t + sw32_chunk_off(r, 0)) = make_uint4(w0, (uint32_t)__half_as_ushort(lo), 0u, 0u);
    *reinterpret_cast<uint4 *>(t + sw32_chunk_off(r, 1)) = make_uint4(0u, 0u, 0u, 0u);
  }
  for (int i = tid; i < H; i += P_THREADS) sWlast[i] = __ldg(prm.W[L - 1] + i) * invS;   // exact: S is a power of two
  const float b_last = __ldg(prm.b[L - 1]);
  fence_async_smem();
  __syncthreads();                                            // the barrier objects are initialised
  mbar_wait_cluster(smem_u32(&bars.wload), 0u);               // the weights have landed
  tc_fence_before();
  cluster.sync();
  tc_fence_after();
  const uint32_t tmem_base = bars.tmem_base_slot;

  const long long npair_tiles = (M + 2 * TC_BM - 1) / (2 * TC_BM);
  const long long nclusters = gridDim.x / 2, cluster_id = blockIdx.x / 2;

  if (warp < P_EPI_WARPS) {
    // =============================== EPILOGUE ===============================
    // Warp q drains TMEM lane quarter q, thread per accumulator row, 32 columns (one tcgen05.ld.x32) at a time with
    // the next 32 in flight.  The accumulator already holds W x + b (the bias K-step).
    //   hidden layer: ReLU + round to fp16 (cvt.rn.relu.f16x2: two elements per instruction) and WRITE THE CHUNK BACK
    //       TO TENSOR MEMORY, in place: the 32 fp32 columns [32c, 32c+32) of the accumulator become the 16 packed
    //       columns [16c, 16c+16) of the same slot (a 32-bit column = two consecutive K elements of the row), which is
    //       the layout tcgen05.mma reads an A operand from — the next layer's MMAs take their A from there and trail
    //       the conversion chunk by chunk (a2_full[c]).  The write position never passes the read position, so no
    //       second buffer is needed, and the activations never touch shared memory: the shared-memory pipe — 128 B
    //       per clock for the gather stores, both MMA operands and, before, 64 KB of activation stores + 64 KB of
    //       A-operand reads per tile — was busy ~85 % of a tile's ideal 4,352 clocks; this takes 128 KB of 384 off it
    //       and frees 48 KB of shared memory for the gather ring.
    //   output layer: ReLU + H -> 1 dot with warp-uniform 128-bit weight loads + sigmoid.
    TR_DECL(1);
    uint32_t acph = 0;            // bit s = phase parity of acc_full[s]
    uint32_t seq = 0;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    for (long long tile = cluster_id; tile < npair_tiles; tile += nclusters) {
      const long long p0 = tile * (2 * TC_BM) + (long long)cta_rank * TC_BM;
      for (int l = 0; l < nhidden; ++l) {
        const uint32_t slot = seq++ & 1u;
        mbar_wait_cluster(smem_u32(&bars.acc_full[slot]), (acph >> slot) & 1u);
        acph ^= 1u << slot;
        tc_fence_after();
        if (tid == 0) TR(5, l, 0);
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + slot * H;
        // 16-column loads, the next one always in flight (same TMEM read rate as 32-column loads,
        // tools/micro/tmem_ld_bw.cu, at half the registers)
        constexpr int NLD = 2 * NCHUNK;
        uint32_t buf[2][16];
        tmem_ld16_issue(taddr, buf[0]);
        if (l < nhidden - 1) {
#pragma unroll
          for (int c = 0; c < NCHUNK; ++c) {
            uint32_t o[16];
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              const int li = 2 * c + hf;
              tmem_ld_wait16(buf[li & 1]);
              if (li + 1 < NLD) tmem_ld16_issue(taddr + (uint32_t)(li + 1) * 16u, buf[(li + 1) & 1]);
              const uint32_t *v = buf[li & 1];
#pragma unroll
              for (int j = 0; j < 8; ++j) o[hf * 8 + j] = cvt_relu_f16x2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
            }
            tmem_st16(taddr + (uint32_t)c * 16u, o);
            tmem_st_wait();
            // the chunk is in place: the tensor pipe starts (continues) the next layer on it while the remaining
            // columns of this tile are still being converted
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_on_cta(smem_u32(&bars.a2_full[c]), 0);
            if (tid == 0) TR(6, c, 0);
          }
          // the slot is handed back as the NEXT layer's A operand; whoever overwrites it later (an MMA of a later
          // layer / tile) is ordered behind the MMAs that read it by the tensor pipe's program order
          __syncwarp();
          if (lane == 0) mbar_arrive_on_cta(smem_u32(&bars.acc_free[slot]), 0);
          if (tid == 0) TR(7, l, 0);
        } else {
          const float4 *w4 = reinterpret_cast<const float4 *>(sWlast);
          float2 part = make_float2(0.f, 0.f);
#pragma unroll
          for (int li = 0; li < NLD; ++li) {
            tmem_ld_wait16(buf[li & 1]);
            if (li + 1 < NLD) tmem_ld16_issue(taddr + (uint32_t)(li + 1) * 16u, buf[(li + 1) & 1]);
            const uint32_t *v = buf[li & 1];
#pragma unroll
            for (int e = 0; e < 16; e += 4) {
              const float4 wa = w4[(li * 16 + e) >> 2];
              float2 t0 = make_float2(fmaxf(__uint_as_float(v[e + 0]), 0.f), fmaxf(__uint_as_float(v[e + 1]), 0.f));
              float2 t1 = make_float2(fmaxf(__uint_as_float(v[e + 2]), 0.f), fmaxf(__uint_as_float(v[e + 3]), 0.f));
              part = fma_f32x2(t0, make_float2(wa.x, wa.y), part);
              part = fma_f32x2(t1, make_float2(wa.z, wa.w), part);
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_on_cta(smem_u32(&bars.acc_free[slot]), 0);
          if (tid == 0) TR(7, l, 0);
          if (p0 + row < M) {
            const float sc = (part.x + part.y) + b_last;
            score[p0 + row] = apply_sigmoid ? sigmoidf_ref(sc) : sc;
          }
        }
      }
    }
  } else if (warp == P_EPI_WARPS) {
    // =============================== MMA ISSUER (leader CTA, one lane) ===============================
    if (cta_rank == 0 && lane == 0) {   // lanes 1..31 wait at the __syncwarp below (keeps the warp
                                        // converged for the aligned cluster barrier at the end)
      TR_DECL(0);
      // This one thread is the tensor pipe's instruction stream: whatever it executes between two
      // tcgen05.mma is time the pipe idles once its short queue drains.  So nothing is derived per
      // iteration — descriptors are a precomputed 64-bit base plus a small constant (the start-address
      // field counts 16-byte units and never carries out of its 14 bits), ring positions and barrier
      // phases are carried incrementally (no division by the run-time ring depth).
      uint32_t afph = 0;
      const uint64_t dRing = umma_smem_desc_sw64(smem_u32(sRing));
      const uint64_t dW = umma_smem_desc(smem_u32(sW));
      const uint64_t dOnes = umma_smem_desc_sw32(smem_u32(sOnes)), dBias = umma_smem_desc_sw32(smem_u32(sBiasB));
      const uint32_t full0 = smem_u32(&bars.full[0]), empty0 = smem_u32(&bars.empty[0]);
      const uint32_t a2full0 = smem_u32(&bars.a2_full[0]);
      uint32_t stage = 0, stage_ph = 0;        // first-layer ring position / parity of full[stage]
      uint32_t a2_ph = 0;                      // parity of a2_full[*] (each is used once per later layer)
      // Issue order: tile by tile, the layers of a tile alternate between the two accumulator slots (layer l+1
      // trails the epilogue of layer l chunk by chunk, the next tile's first layer overlaps the last epilogue).
      uint32_t seq = 0;
      for (long long tile = cluster_id; tile < npair_tiles; tile += nclusters) {
        for (int l = 0; l < nhidden; ++l) {
          const uint32_t slot = seq++ & 1u;
          mbar_wait_cluster(smem_u32(&bars.acc_free[slot]), ((afph >> slot) & 1u) ^ 1u);   // first use passes
          afph ^= 1u << slot;
          tc_fence_after();
          TR(1, l, 0);
          const uint32_t d = tmem_base + slot * H;
          // bias K-step: initialises the accumulator with b[l] in every row
          umma_f16_ss_2cta_p(d, dOnes, dBias + (uint64_t)(l * ((HH * 32) >> 4)), IDESC, 0u);
          const uint64_t dWl = dW + (uint64_t)(l * (WH_BYTES >> 4));
          // The barrier of the NEXT chunk is looked at right after the first MMA of the current one has been
          // issued, so its round trip to shared memory runs under that MMA instead of between two of them.
          uint32_t ready = 0;
          if (l == 0) {
#pragma unroll
            for (int c = 0; c < NCHUNK; ++c) {
              if (!ready) mbar_wait_cluster(full0 + stage * 8u, stage_ph);
              tc_fence_after();
              TR(2, c, 0);
              const uint64_t ad = dRing + (uint64_t)(stage * (P_STAGE_BYTES >> 4));
              const uint32_t cur = stage;
              if (++stage == (uint32_t)ring) { stage = 0; stage_ph ^= 1u; }
#pragma unroll
              for (int k16 = 0; k16 < P_CHUNK_K / 16; ++k16) {
                const int k = c * P_CHUNK_K + k16 * 16;
                umma_f16_ss_2cta_p(d, ad + (uint64_t)(k16 * 2),
                                    dWl + (uint64_t)(((k >> 6) * (HH * 128) + ((k & 63) >> 4) * 32) >> 4), IDESC, 1u);
                if (k16 == 0) ready = (c + 1 < NCHUNK) ? mbar_test(full0 + stage * 8u, stage_ph) : 0u;
              }
              umma_commit_mc(empty0 + cur * 8u);            // stage reusable once these MMAs retire
            }
          } else {
            // A operand = the previous layer's activations, fp16-packed in the OTHER accumulator slot (see the epilogue)
            const uint32_t a_tmem = tmem_base + (slot ^ 1u) * H;
#pragma unroll
            for (int c = 0; c < NCHUNK; ++c) {
              if (!ready) mbar_wait_cluster(a2full0 + (uint32_t)c * 8u, a2_ph);   // chunk c has been converted
              tc_fence_after();
              TR(3, c, 0);
#pragma unroll
              for (int k16 = 0; k16 < P_CHUNK_K / 16; ++k16) {
                const int k = c * P_CHUNK_K + k16 * 16;
                umma_f16_ts_2cta_p(d, a_tmem + (uint32_t)(k >> 1),
                                    dWl + (uint64_t)(((k >> 6) * (HH * 128) + ((k & 63) >> 4) * 32) >> 4), IDESC, 1u);
                if (k16 == 0) ready = (c + 1 < NCHUNK) ? mbar_test(a2full0 + (uint32_t)(c + 1) * 8u, a2_ph) : 0u;
              }
            }
            a2_ph ^= 1u;
          }
          umma_commit_mc(smem_u32(&bars.acc_full[slot]));
          TR(4, l, 0);
        }
      }
    }
    __syncwarp();
  } else if (warp == P_IDS_WARP) {
    // =============================== PAIR IDS ===============================
    // (u, v) of this CTA's 128 rows -> shared memory, one tile ahead of the warps that gather, so a row gather never
    // waits on a dependent index load.  Tiles run in list order: a u-blocked order that keeps a node range's rows in
    // L2 was measured slower (profiles/round1_e_k2_tile_schedule.md).  The ids of the tile after that are already in
    // registers; on the fp32-source path their embedding rows are pulled into L2 from there (one DRAM page visit per
    // row instead of one per chunk-sized piece; the gathers, about one tile-time later, then hit L2).  The fp16-table
    // path has no prefetch: its loaders run a ring ahead themselves, and the prefetch cost 2-4 % there
    // (profiles/round2_d_k2_timeline.md, steps 10-11).
    constexpr int RB = H * (HB ? 2 : 4);
    const char *hb = reinterpret_cast<const char *>(h);
    int nu[4], nv[4];
    auto load_ids = [&](long long tile) {
      const long long p0 = tile * (2 * TC_BM) + (long long)cta_rank * TC_BM;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const long long p = p0 + lane + 32 * q;
        nu[q] = -1; nv[q] = -1;
        if (p < M) { nu[q] = __ldg(pu + p); nv[q] = __ldg(pv + p); }
      }
      if constexpr (!HB) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int vprev = __shfl_up_sync(FULL, nv[q], 1);
          if (nu[q] >= 0) {
            const char *rup = hb + (size_t)nu[q] * RB;
#pragma unroll
            for (int b = 0; b < RB; b += 128) asm volatile("prefetch.global.L2 [%0];" :: "l"(rup + b));
            if (lane == 0 || vprev != nv[q]) {                   // runs of equal v: prefetch each row once
              const char *rvp = hb + (size_t)nv[q] * RB;
#pragma unroll
              for (int b = 0; b < RB; b += 128) asm volatile("prefetch.global.L2 [%0];" :: "l"(rvp + b));
            }
          }
        }
      }
    };
    if (cluster_id < npair_tiles) load_ids(cluster_id);
    long long tl = 0;
    for (long long tile = cluster_id; tile < npair_tiles; tile += nclusters, ++tl) {
      const int slot = (int)(tl & 1);
      mbar_wait_cluster(smem_u32(&bars.ids_empty[slot]), (uint32_t)(((tl >> 1) & 1) ^ 1));
#pragma unroll
      for (int q = 0; q < 4; ++q) sIds[slot * TC_BM + lane + 32 * q] = make_int2(nu[q], nv[q]);
      if constexpr (HB) {
        // The h[v] rows of the tile's owners go to shared memory ONCE per tile (the rows are grouped by v: a tile has
        // one owner, now and then two), so the warps that multiply never load from global memory: a register load of
        // the h[v] piece per chunk, even an L1/L2 hit, sat in their dependency chain with 400-500 clocks
        // (profiles/round2_d_k2_timeline.md).  Row r gets the index of its owner's row in sV, or -1 beyond P_VROWS
        // owners (arbitrary pair lists: those rows fall back to a global load).
        int carry = 0, last_v = -2;
        int kq[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          int vprev = __shfl_up_sync(FULL, nv[q], 1);
          if (lane == 0) vprev = last_v;
          const bool flag = nu[q] >= 0 && nv[q] != vprev;
          const unsigned bal = __ballot_sync(FULL, flag);
          const int k = carry + __popc(bal & (0xffffffffu >> (31 - lane))) - 1;
          if (flag && k < P_VROWS) sVid[k] = nv[q];
          kq[q] = (nu[q] >= 0 && k >= 0 && k < P_VROWS) ? k : -1;
          carry += __popc(bal);
          last_v = __shfl_sync(FULL, nv[q], 31);
        }
        __syncwarp();
        const int nd = min(carry, P_VROWS);
        for (int k = 0; k < nd; ++k) {
          if (lane < H * 2 / 16) {
            const char *src = hb + (size_t)sVid[k] * RB + lane * 16;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                         :: "r"(smem_u32(sV + ((size_t)slot * P_VROWS + k) * (H * 2) + lane * 16)), "l"(src) : "memory");
          }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
#pragma unroll
        for (int q = 0; q < 4; ++q) sKi[slot * TC_BM + lane + 32 * q] = kq[q];
        if (tile + nclusters < npair_tiles) load_ids(tile + nclusters);     // in flight while the rows land
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive_on_cta(smem_u32(&bars.ids_full[slot]), cta_rank);
      } else {
        __syncwarp();
        if (lane == 0) mbar_arrive_on_cta(smem_u32(&bars.ids_full[slot]), cta_rank);
        if (tile + nclusters < npair_tiles) load_ids(tile + nclusters);
      }
    }
  } else if (NL > 0 && warp < P_FIRST_PROD_WARP) {
   if constexpr (NL > 0) {
    // =============================== LOADERS (fp16 table) ===============================
    // The gather is LATENCY bound (a 64-byte piece of a random row takes ~1,400 clocks under load), so it is done by
    // warps that never wait for data: cp.async (LDGSTS) of the h[u] pieces of chunk j straight into ring stage
    // j % ring, at their SWIZZLE_64B position, and the copies arrive on the stage's `landed` barrier themselves
    // (cp.async.mbarrier.arrive.noinc).  The whole ring — all the shared memory the resident weights leave — is in
    // flight ahead of the tensor pipe.  Dedicated warps because (a) LDGSTS bandwidth of such pieces scales with the
    // number of issuing warps (1 warp: 2-5 B/clk, 4: 7-24, 8: 13-47; tools/micro/gather_bw.cu), and (b) the warps
    // that MULTIPLY the landed pieces must fence.proxy.async before the MMA may read them, and that fence waits for
    // the executing thread's own outstanding cp.async — issued by the same threads, the copies of the next chunks
    // would be drained at every hand-off (measured: 700-1,400 clocks per chunk, profiles/round2_d_k2_timeline.md).
    // Lane (r8 = lane / 4, l4 = lane % 4) of loader warp w copies unit l4 of rows r8 + 8 (w + NL j), j < 16 / NL.
    constexpr int RPL = 16 / (NL > 0 ? NL : 1);
    TR_DECL(6);
    const int lw = warp - P_FIRST_LOAD_WARP, r8 = lane >> 2, l4 = lane & 3;
    const char *hb = reinterpret_cast<const char *>(h);
    long long my_tiles = 0;
    if (cluster_id < npair_tiles) my_tiles = (npair_tiles - cluster_id + nclusters - 1) / nclusters;
    uint32_t stage = 0, eph = 1u;                              // ring position / parity its `empty` barrier is waited with
    for (long long tl = 0; tl < my_tiles; ++tl) {
      const int slot = (int)(tl & 1);
      mbar_wait_cluster(smem_u32(&bars.ids_full[slot]), (uint32_t)((tl >> 1) & 1));
      int ru[RPL];
#pragma unroll
      for (int j = 0; j < RPL; ++j) ru[j] = sIds[slot * TC_BM + r8 + 8 * (lw + NL * j)].x;
      __syncwarp();
      if (lane == 0) mbar_arrive_on_cta(smem_u32(&bars.ids_empty[slot]), cta_rank);     // the ids are in registers
#pragma unroll 1
      for (int c = 0; c < NCHUNK; ++c) {
        mbar_wait_cluster(smem_u32(&bars.empty[stage]), eph);              // the MMAs that read this stage retired
        const uint32_t dst0 = smem_u32(sRing + stage * P_STAGE_BYTES);
        const int boff = (c * P_CHUNK_K + l4 * 8) * 2;
#pragma unroll
        for (int j = 0; j < RPL; ++j) {
          const bool ok = ru[j] >= 0;
          const char *src = hb + (ok ? (size_t)ru[j] * (H * 2) + boff : (size_t)0);
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;"
                       :: "r"(dst0 + sw64_chunk_off(r8 + 8 * (lw + NL * j), l4)), "l"(src), "r"(ok ? 16 : 0) : "memory");   // 0: zero fill
        }
        asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" :: "r"(smem_u32(&bars.landed[stage])) : "memory");
        if (lw == 0 && lane == 0) TR(8, c, 0);
        if (++stage == (uint32_t)ring) { stage = 0; eph ^= 1u; }
      }
    }
   }
  } else {
    // =============================== PRODUCERS ===============================
    // NG independent groups of four warps; group g produces chunks g, g+NG, g+2NG, ... of the flattened chunk
    // stream of this CTA's tiles (a chunk = 128 rows x 32 K) in ring stage (chunk % ring).
    // Lane mapping inside a group (128 threads): 4 consecutive lanes cover one row's chunk, each lane
    // 8 K-elements = one 16-byte unit of the swizzled stage; a warp instruction covers 8 rows.
    //   fp16 table (the hot path): the h[u] pieces are ALREADY in the stage (cp.async, see the loader warps); the
    //       group multiplies them in place by h[v] — one 16-byte piece per thread and chunk, because the list is
    //       grouped by v (a row whose v differs fetches its own piece, predicated) — and hands the stage to the MMA;
    //   fp32 source (short pair lists, no table): 4 x LDG.128 per row into registers, rounded like the table.
    const int pw = warp - P_FIRST_PROD_WARP;
    const int group = pw / P_GROUP_WARPS;
    const int t = (pw % P_GROUP_WARPS) * 32 + lane;          // 0..127
    const int l4 = t & 3;
    const int rg = t >> 2;                                   // 0..31 ; rows rg + 32 q, q < 4
    long long my_tiles = 0;
    if (cluster_id < npair_tiles) my_tiles = (npair_tiles - cluster_id + nclusters - 1) / nclusters;
    const long long total = my_tiles * NCHUNK;
    const char *hbase = reinterpret_cast<const char *>(h);
    constexpr int ROW_BYTES = H * (HB ? 2 : 4);
    long long cur_tl = -1;
    int idu[4], idv[4];
    TR_DECL(2 + group);
    // Move this warp's position in the pair-id pipeline to tile `tl`: release every tile left behind
    // (also tiles this group has no chunk in — H = 64 has 2 chunks per tile for 3 groups), waiting
    // for each tile's ids to have been published first so that a release can never be counted
    // towards an earlier phase of the same slot.
    auto advance_to = [&](long long tl) {
      while (cur_tl < tl) {
        if (cur_tl >= 0) {
          __syncwarp();
          if (lane == 0) mbar_arrive_on_cta(smem_u32(&bars.ids_empty[cur_tl & 1]), cta_rank);
        }
        ++cur_tl;
        if (cur_tl < my_tiles)
          mbar_wait_cluster(smem_u32(&bars.ids_full[cur_tl & 1]), (uint32_t)((cur_tl >> 1) & 1));
      }
    };
    auto enter_tile = [&](long long tl) {
      advance_to(tl);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int2 id = sIds[(tl & 1) * TC_BM + rg + 32 * q];
        idu[q] = id.x; idv[q] = id.y;
      }
    };
    // ring position of this group's next chunk and the parities its barriers are waited with, carried
    // incrementally (the group's chunks are NG apart and NG < ring: at most one wrap a step)
    uint32_t pstage = (uint32_t)group;
    if constexpr (HB) {
      // fp16 table: the h[u] pieces of chunk i are ALREADY in stage i % ring (the loader warps); this group multiplies
      // them in place by h[v] — read from the tile's staged owner rows in shared memory (the ids warp), so nothing in
      // this loop waits on global memory — and hands the stage to the MMA issuer.
      uint32_t lphase = 0u;                                    // parity landed[pstage] is waited with
      int kq[4] = {-1, -1, -1, -1};
      bool uni = false;
      const uint8_t *sVt = sV;
      for (long long i = group; i < total; i += NG) {
        const long long tl = i / NCHUNK;
        const int c = (int)(i - tl * NCHUNK);
        if (tl != cur_tl) {
          enter_tile(tl);
#pragma unroll
          for (int q = 0; q < 4; ++q) kq[q] = sKi[(tl & 1) * TC_BM + rg + 32 * q];
          sVt = sV + (size_t)(tl & 1) * P_VROWS * (H * 2);
          // rows beyond the list (u < 0) were zero-filled by the copy: 0 * anything finite = 0, they may share the path
          uni = kq[0] >= 0;
#pragma unroll
          for (int q = 1; q < 4; ++q) uni = uni && (kq[q] == kq[0] || idu[q] < 0);
        }
        const int boff = (c * P_CHUNK_K + l4 * 8) * 2;
        const uint32_t stage = pstage;
        mbar_wait_cluster(smem_u32(&bars.landed[stage]), lphase);        // the gathered pieces have landed
        pstage += NG;
        if (pstage >= (uint32_t)ring) { pstage -= (uint32_t)ring; lphase ^= 1u; }
        if (t == 0) TR(9, c, group);
        uint8_t *dst = sRing + stage * P_STAGE_BYTES;
        if (uni) {
          // the thread's four rows share one staged owner row (almost always): all five shared-memory loads are issued
          // before the first multiply, so the chunk costs ONE load latency, not four in a row
          const uint4 xv = *reinterpret_cast<const uint4 *>(sVt + kq[0] * (H * 2) + boff);       // warp-wide broadcast
          uint4 xu[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) xu[q] = *reinterpret_cast<const uint4 *>(dst + sw64_chunk_off(rg + 32 * q, l4));
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint4 o;
            o.x = mul_f16x2(xu[q].x, xv.x); o.y = mul_f16x2(xu[q].y, xv.y);
            o.z = mul_f16x2(xu[q].z, xv.z); o.w = mul_f16x2(xu[q].w, xv.w);
            *reinterpret_cast<uint4 *>(dst + sw64_chunk_off(rg + 32 * q, l4)) = o;      // tail rows were zero-filled by the copy
          }
        } else {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint4 *cell = reinterpret_cast<uint4 *>(dst + sw64_chunk_off(rg + 32 * q, l4));
            const uint4 xu = *cell;
            uint4 xv;
            if (kq[q] >= 0) xv = *reinterpret_cast<const uint4 *>(sVt + kq[q] * (H * 2) + boff);
            else xv = __ldg(reinterpret_cast<const uint4 *>(hbase + (size_t)max(idv[q], 0) * ROW_BYTES + boff));
            uint4 o;
            o.x = mul_f16x2(xu.x, xv.x); o.y = mul_f16x2(xu.y, xv.y);
            o.z = mul_f16x2(xu.z, xv.z); o.w = mul_f16x2(xu.w, xv.w);
            if (idu[q] < 0) o = make_uint4(0u, 0u, 0u, 0u);
            *cell = o;
          }
        }
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive_on_cta(smem_u32(&bars.full[stage]), 0);
        if (t == 0) TR(10, c, group);
      }
    } else {
      uint32_t ephase = 1u;
      for (long long i = group; i < total; i += NG) {
        const long long tl = i / NCHUNK;
        const int c = (int)(i - tl * NCHUNK);
        if (tl != cur_tl) enter_tile(tl);
        const int boff = (c * P_CHUNK_K + l4 * 8) * 4;
        uint4 xu[4][2], xv[2];
        xv[0] = xv[1] = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          xu[q][0] = xu[q][1] = make_uint4(0u, 0u, 0u, 0u);
          if (idu[q] >= 0) {
            const uint4 *pu4 = reinterpret_cast<const uint4 *>(hbase + (size_t)idu[q] * ROW_BYTES + boff);
            xu[q][0] = __ldg(pu4); xu[q][1] = __ldg(pu4 + 1);
          }
        }
        if (idu[0] >= 0) {
          const uint4 *pv4 = reinterpret_cast<const uint4 *>(hbase + (size_t)idv[0] * ROW_BYTES + boff);
          xv[0] = __ldg(pv4); xv[1] = __ldg(pv4 + 1);
        }
        const uint32_t stage = pstage;
        mbar_wait_cluster(smem_u32(&bars.empty[stage]), ephase);   // the MMAs that read this stage retired
        pstage += NG;
        if (pstage >= (uint32_t)ring) { pstage -= (uint32_t)ring; ephase ^= 1u; }
        uint8_t *dst = sRing + stage * P_STAGE_BYTES;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 c0 = xv[0], c1 = xv[1];
          if (q > 0 && idu[q] >= 0 && idv[q] != idv[0]) {
            const uint4 *pv4 = reinterpret_cast<const uint4 *>(hbase + (size_t)idv[q] * ROW_BYTES + boff);
            c0 = __ldg(pv4); c1 = __ldg(pv4 + 1);
          }
          const uint4 a0 = xu[q][0], a1 = xu[q][1];
          uint4 o;
          o.x = hadamard_f16x2(__uint_as_float(a0.x), __uint_as_float(a0.y), __uint_as_float(c0.x), __uint_as_float(c0.y), hscale);
          o.y = hadamard_f16x2(__uint_as_float(a0.z), __uint_as_float(a0.w), __uint_as_float(c0.z), __uint_as_float(c0.w), hscale);
          o.z = hadamard_f16x2(__uint_as_float(a1.x), __uint_as_float(a1.y), __uint_as_float(c1.x), __uint_as_float(c1.y), hscale);
          o.w = hadamard_f16x2(__uint_as_float(a1.z), __uint_as_float(a1.w), __uint_as_float(c1.z), __uint_as_float(c1.w), hscale);
          if (idu[q] < 0) o = make_uint4(0u, 0u, 0u, 0u);
          *reinterpret_cast<uint4 *>(dst + sw64_chunk_off(rg + 32 * q, l4)) = o;
        }
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive_on_cta(smem_u32(&bars.full[stage]), 0);
      }
    }
    advance_to(my_tiles);                                    // release the tiles this group had no chunk in
  }
  tc_fence_before();
  cluster.sync();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

template <int H, bool HB>
static int tc3_launch(const void *h, const int *pu, const int *pv, long long M, const MlpParams &prm, int L,
                      int apply_sigmoid, float *score, uint8_t *img, const TcScale *scale, cudaStream_t stream) {
  const int nhidden = L - 1;
  const size_t fixed = (size_t)nhidden * (H / 2) * H * 2 +
                       (size_t)TC_BM * 32 + (size_t)nhidden * (H / 2) * 32 +          // bias K-step tiles
                       sizeof(float) * (size_t)H + 2 * TC_BM * sizeof(int2) + 2 * TC_BM * sizeof(int) +
                       (HB ? (size_t)2 * P_VROWS * H * 2 : 0) + 32 + sizeof(PipeBarriers);
  const size_t budget = 227 * 1024;
  if (fixed + (size_t)(p_groups(HB) + 1) * P_STAGE_BYTES > budget) return EPS_ERR_UNSUPPORTED;   // the resident weights do not fit (H = 256, L >= 4)
  const int ring = (int)std::min<size_t>((budget - fixed) / P_STAGE_BYTES, (size_t)P_MAX_RING);
  const size_t smem = fixed + (size_t)ring * P_STAGE_BYTES;
  auto kern = linkpred_tc3_kernel<H, HB>;
  EPS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long npair_tiles = (M + 2 * TC_BM - 1) / (2 * TC_BM);
  const int clusters = (int)std::min<long long>(npair_tiles, (long long)(sm_count() / 2));
  kern<<<2 * clusters, p_threads(HB), smem, stream>>>(h, pu, pv, M, prm, L, apply_sigmoid, img, score, ring, scale);
  EPS_LAUNCH_CHECK();
#ifdef EPS_TC3_TRACE
  if (const char *tf = getenv("EPS_TC3_TRACE_FILE")) {
    cudaStreamSynchronize(stream);
    std::vector<unsigned long long> rec(8 * TR_REGION);
    cudaMemcpyFromSymbol(rec.data(), g_trace, rec.size() * 8);
    if (FILE *f = fopen(tf, "wb")) { fwrite(rec.data(), 8, rec.size(), f); fclose(f); }
    std::fill(rec.begin(), rec.end(), 0ull);
    cudaMemcpyToSymbol(g_trace, rec.data(), rec.size() * 8);
  }
#endif
  return EPS_OK;
}

// ---- prepare kernels: scale, fp16 table, weight images (once per (h, weights); EPS_MLP_REUSE_WORKSPACE skips them) ----

// max |h| as the bit pattern of a non-negative float (orders like an unsigned integer)
__global__ void __launch_bounds__(256) tc_absmax_kernel(const float *__restrict__ h, long long n4, unsigned int *out_bits) {
  float m = 0.f;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = __ldg(reinterpret_cast<const float4 *>(h) + i);
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(FULL, m, o));
  if (lane_id() == 0) atomicMax(out_bits, __float_as_uint(m));
}

// The power-of-two scale of the arm (tc_common.cuh).  Worst-case magnitudes, unscaled:
//   products     P   = hmax^2
//   layer l out  B_l = (max_n sum_k |W_l[n,k]|) * B_{l-1} + max_n |b_l[n]|,   B_0 = P
// and S = hscale^2 = 4^a is the largest power of four with S * max(P, B_1, ..) <= 2^15 (half of fp16's largest
// finite value), so no operand can overflow; typical magnitudes sit 10^2..10^4 below the worst case, well inside
// fp16's normal range.  One block.
__global__ void __launch_bounds__(256) tc_scale_kernel(const unsigned int *__restrict__ hmax_bits, const MlpParams prm,
                                                       int H, int nhidden, TcScale *out) {
  __shared__ double red[256];
  const int t = threadIdx.x;
  const float hmax = __uint_as_float(*hmax_bits);
  double bound = (double)hmax * (double)hmax, worst = bound;
  for (int l = 0; l < nhidden; ++l) {
    double row = 0.0, bm = 0.0;
    for (int n = t; n < H; n += 256) {
      double acc = 0.0;
      for (int k = 0; k < H; ++k) acc += fabs((double)__ldg(prm.W[l] + (size_t)n * H + k));
      row = fmax(row, acc);
      bm = fmax(bm, fabs((double)__ldg(prm.b[l] + n)));
    }
    red[t] = row;
    __syncthreads();
    for (int o = 128; o; o >>= 1) { if (t < o) red[t] = fmax(red[t], red[t + o]); __syncthreads(); }
    const double rmax = red[0];
    __syncthreads();
    red[t] = bm;
    __syncthreads();
    for (int o = 128; o; o >>= 1) { if (t < o) red[t] = fmax(red[t], red[t + o]); __syncthreads(); }
    const double bmax = red[0];
    __syncthreads();
    bound = rmax * bound + bmax;
    worst = fmax(worst, bound);
  }
  if (t == 0) {
    int a = 0;
    if (worst > 0.0 && worst < 1e300) a = (int)floor(log2(32768.0 / worst) * 0.5);
    a = max(-40, min(40, a));
    out->hscale = exp2f((float)a);
    out->S = exp2f((float)(2 * a));
    out->invS = exp2f((float)(-2 * a));
    out->hmax = hmax;
  }
}

// fp32 embeddings -> fp16 table of h * hscale (round to nearest even), 8 elements per thread
__global__ void __launch_bounds__(256) h_to_f16_kernel(const float *__restrict__ h, long long n8, const TcScale *__restrict__ scale,
                                                       uint4 *__restrict__ out) {
  const float hs = scale->hscale;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
    const float4 a = __ldg(reinterpret_cast<const float4 *>(h) + 2 * i);
    const float4 b = __ldg(reinterpret_cast<const float4 *>(h) + 2 * i + 1);
    uint4 o;
    o.x = pack_f16x2(a.x * hs, a.y * hs); o.y = pack_f16x2(a.z * hs, a.w * hs);
    o.z = pack_f16x2(b.x * hs, b.y * hs); o.w = pack_f16x2(b.z * hs, b.w * hs);
    out[i] = o;
  }
}

// hidden-layer weights -> per-CTA-half fp16 SWIZZLE_128B images: [layer][half][kblock][H/2 rows][128 B]
__global__ void pack_weights_halves_kernel(MlpParams prm, int H, int nhidden, uint8_t *img) {
  const int chunks_per_row = H / 8, HH = H / 2;
  const int total = nhidden * H * chunks_per_row;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int l = i / (H * chunks_per_row);
    const int rem = i - l * H * chunks_per_row;
    const int n = rem / chunks_per_row, c = rem - n * chunks_per_row;
    const float *w = prm.W[l] + (size_t)n * H + c * 8;
    const float4 a = *reinterpret_cast<const float4 *>(w), b = *reinterpret_cast<const float4 *>(w + 4);
    uint4 o;
    o.x = pack_f16x2(a.x, a.y); o.y = pack_f16x2(a.z, a.w);
    o.z = pack_f16x2(b.x, b.y); o.w = pack_f16x2(b.z, b.w);
    const int half = n / HH, nn = n - half * HH;
    *reinterpret_cast<uint4 *>(img + (size_t)l * H * H * 2 + (size_t)half * HH * H * 2 +
                               sw128_chunk_off(HH, nn, c * 8)) = o;
  }
}

// The kernel gathers from an fp16 copy of h (half the bytes per pair) when the pair list is long enough to
// amortise writing it; short lists read the caller's fp32 rows and round them in registers — the SAME
// rounding, so the scores do not depend on this choice.
bool linkpred_tc_uses_table(int n, long long M) { return M >= 2ll * n; }

static size_t tc_img_bytes(int H, int L) {
  return ((size_t)std::max(L - 1, 0) * H * H * 2 + 255) & ~(size_t)255;
}

size_t linkpred_tc_workspace_bytes(int n, int H, int L, long long M) {
  // header (TcScale, max |h|) | weight images | fp16 embedding table: on the table path the size does not depend on M
  return 256 + tc_img_bytes(H, L) + (linkpred_tc_uses_table(n, M) ? (((size_t)n * H * 2 + 255) & ~(size_t)255) : 0);
}

int linkpred_tc_launch(const float *h, int n, int H, const int *pu, const int *pv, long long M,
                       const MlpParams &prm, int L, int apply_sigmoid, float *score, void *workspace,
                       size_t workspace_bytes, bool prepared, cudaStream_t stream) {
  if (L < 2 || !(H == 64 || H == 128 || H == 256) || (H == 256 && L > 3)) {
    set_error("eps_linkpred_mlp: the tcgen05 arm needs num_layers >= 2, H in {64,128,256} and its hidden-layer weights "
              "resident in shared memory (H = 256: num_layers <= 3) (got L=%d H=%d); use EPS_MLP_FP32", L, H);
    return EPS_ERR_UNSUPPORTED;
  }
  if (!workspace || workspace_bytes < linkpred_tc_workspace_bytes(n, H, L, M)) {
    set_error("eps_linkpred_mlp: workspace too small");
    return EPS_ERR_WORKSPACE;
  }
  uint8_t *ws = (uint8_t *)workspace;
  TcScale *scale = (TcScale *)ws;
  unsigned int *hmax_bits = (unsigned int *)(ws + 64);
  uint8_t *img = ws + 256;
  const bool use_table = linkpred_tc_uses_table(n, M);
  void *table = use_table ? img + tc_img_bytes(H, L) : nullptr;
  if (!prepared) {                                  // EPS_MLP_REUSE_WORKSPACE: scale, table and images are still there
    const int sms = sm_count();
    EPS_CUDA(cudaMemsetAsync(hmax_bits, 0, 4, stream));
    const long long n4 = (long long)n * H / 4;
    tc_absmax_kernel<<<(int)std::min<long long>((n4 + 255) / 256, (long long)sms * 16), 256, 0, stream>>>(h, n4, hmax_bits);
    tc_scale_kernel<<<1, 256, 0, stream>>>(hmax_bits, prm, H, L - 1, scale);
    if (use_table) {
      const long long n8 = (long long)n * H / 8;
      h_to_f16_kernel<<<(int)std::min<long long>((n8 + 255) / 256, (long long)sms * 16), 256, 0, stream>>>(
          h, n8, scale, reinterpret_cast<uint4 *>(table));
    }
    const int total = (L - 1) * H * (H / 8);
    pack_weights_halves_kernel<<<(total + 255) / 256, 256, 0, stream>>>(prm, H, L - 1, img);
    EPS_LAUNCH_CHECK();
  }
#define EPS_TC3(HV)                                                                                           \
  return use_table ? tc3_launch<HV, true>(table, pu, pv, M, prm, L, apply_sigmoid, score, img, scale, stream) \
                   : tc3_launch<HV, false>(h, pu, pv, M, prm, L, apply_sigmoid, score, img, scale, stream)
  if (H == 64) { EPS_TC3(64); }
  if (H == 128) { EPS_TC3(128); }
  EPS_TC3(256);
#undef EPS_TC3
}

}  // namespace eps
