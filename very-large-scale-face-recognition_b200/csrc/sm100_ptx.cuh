// Inline-PTX wrappers (mbarrier, TMA, tcgen05 / TMEM, cluster) and the register-resident hard-negative top-k helpers shared by the
// two tcgen05 sweep kernels (head_sm100.cu: CTA pair, any D up to 512; head_sm100_1cta.cu: one CTA, D <= 256).  sm_100a only.
#pragma once
#include <cuda.h>

#include "head_internal.cuh"

namespace ffc {

constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t remote_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_addr) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(addr),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {   // pairs with a remote release.cluster arrive
  const uint32_t addr = smem_u32(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAITC_LOOP:\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAITC_DONE;\n"
      "bra WAITC_LOOP;\n"
      "WAITC_DONE:\n"
      "}\n" ::"r"(addr),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ uint32_t map_to_rank(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int x, int y) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
               "l"(map), "r"(smem_u32(bar)), "r"(x), "r"(y)
               : "memory");
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* map, uint64_t* bar, void* dst, int x, int y, int z) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(dst)),
               "l"(map), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]),
      "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]),
      "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
        "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
        "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
        "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// asynchronous 16-byte store into the peer CTA's shared memory; completion is counted (complete_tx) on the
// peer's mbarrier, so the writer needs no fence / drain before the consumer may be released
__device__ __forceinline__ void st_async_v4(uint32_t addr, uint32_t mbar, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(addr), "r"(a), "r"(b),
               "r"(c), "r"(d), "r"(mbar)
               : "memory");
}
// tcgen05.commit that arrives on the barrier at the same offset in the CTAs of `cta_mask`
__device__ __forceinline__ void tc_commit_mcast(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}

// UMMA shared-memory descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor): SWIZZLE_128B, version 1
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type = 2) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
  d |= (uint64_t)1 << 46;   // version = 1 (Blackwell)
  d |= (uint64_t)layout_type << 61;   // 2 = SWIZZLE_128B, 0 = SWIZZLE_NONE (interleaved 8x16-byte core matrices)
  return d;
}
// instruction descriptor (InstrDescriptor): bf16 x bf16 -> f32
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

// One lane of a converged warp; the warp stays converged, so descriptors live in uniform registers and consecutive
// tcgen05.mma issue back to back.  (Issuing from an `if (lane == 0)` region makes every MMA pay a vote loop plus
// register->uniform moves: 125-220 cycles per instruction against the 64 / 128 cycles the tensor pipe needs.)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile("{\n.reg .pred px;\nelect.sync _|px, 0xffffffff;\nselp.u32 %0, 1, 0, px;\n}\n" : "=r"(pred));
  return pred != 0;
}

constexpr uint32_t TOPK_VAL_MASK = 0xffffffe0u;   // top-k keys: cosine bits with the low 5 mantissa bits replaced by the column's index in its chunk

__device__ __forceinline__ uint32_t max_bf16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}

// Hard-negative top-k (ffc.py:86-92) over 16 raw cosines v[BASE .. BASE+16) of one row (= lane), columns col0 .. col0+15.
// Branch-free register list of integer keys: only POSITIVE cosines can contribute (clip(.., 0) zeroes the rest and their
// gradient), positive floats order like their int32 bit patterns, and the low 4 mantissa bits carry the column's index inside
// the chunk (5 bits: up to 32 columns; value error 2^-18).  tk[] descending keys (0 = empty), tc[] first column of the chunk a key came from.
// Warp-collective: all lanes run the same code; a lane with a candidate (key above its threshold `kth`) extracts its largest
// remaining key per round until no lane has any left.  `kfloor` is the row's threshold shared by the column chunks (below).
// SIGNED (identification, cosines of any sign): the keys are topk_ord() of the cosine bits instead, and INT_MIN means empty.
// sorted insertion of one key into the branch-free register list (the caller has checked xk > kth)
__device__ __forceinline__ void topk_insert_key(int xk, int xc, int k, int (&tk)[KMAX], int (&tc)[KMAX]) {
#pragma unroll
  for (int r = 0; r < KMAX; ++r) {
    if (r < k) {
      const bool pgt = xk > tk[r];
      const int nk = pgt ? xk : tk[r], nc = pgt ? xc : tc[r];
      xk = pgt ? tk[r] : xk;
      xc = pgt ? tc[r] : xc;
      tk[r] = nk;
      tc[r] = nc;
    }
  }
}

// order-preserving map of float bits to int32 (any sign): x < y  <=>  topk_ord(x) < topk_ord(y)
__host__ __device__ __forceinline__ int topk_ord(uint32_t bits) { return (int)bits >= 0 ? (int)bits : (int)(bits ^ 0x7fffffffu); }

template <int BASE, int NV, bool SIGNED = false>
__device__ __forceinline__ void topk_scan16(const uint32_t (&v)[NV], uint32_t excl, int col0, bool outl, int k, int (&tk)[KMAX], int (&tc)[KMAX],
                                            int& kth, int kfloor) {
  constexpr int EMPTY = SIGNED ? (int)0x80000000u : 0;
  int key[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) {
    key[c] = (int)(((SIGNED ? (uint32_t)topk_ord(v[BASE + c]) : v[BASE + c]) & TOPK_VAL_MASK) | (uint32_t)c);
    if ((excl >> c) & 1u) key[c] = EMPTY;
  }
  int bound = 0x7fffffff;      // keys >= bound were already extracted in this chunk
  while (true) {
    int mx = EMPTY;
#pragma unroll
    for (int c = 0; c < 16; ++c) mx = max(mx, key[c] < bound ? key[c] : EMPTY);
    const bool has = outl && mx > kth;
    if (!__any_sync(0xffffffffu, has)) break;
    if (has) {
      int xk = mx, xc = col0;
#pragma unroll
      for (int r = 0; r < KMAX; ++r) {
        if (r < k) {
          const bool pgt = xk > tk[r];
          const int nk = pgt ? xk : tk[r], nc = pgt ? xc : tc[r];
          xk = pgt ? tk[r] : xk;
          xc = pgt ? tc[r] : xc;
          tk[r] = nk;
          tc[r] = nc;
        }
      }
#pragma unroll
      for (int r = 0; r < KMAX; ++r)
        if (r == k - 1) kth = max(tk[r], kfloor);     // own k-th, or the row's shared threshold if that is higher
      bound = mx;
    } else {
      bound = EMPTY;           // this lane is done with the chunk
    }
  }
}

// One launch runs up to MAX_SUB sweeps that share the probe rows P (their work items are concatenated): the main sweep over
// queue[0] and the two tiny side sweeps over the gathered `ones` rows.  The main sweep of C3 fills 72 of the 74 CTA-pair
// slots, so the side items run on the two spare pairs while it is in flight instead of as two more launches.
constexpr int MAX_SUB = 3;
struct SubSweep {
  int64_t n_cols;
  const int32_t* n_cols_dev;
  const int32_t* tcol;
  const uint32_t* cmask;
  const float* thr;
  int tiles_per_chunk;
  int n_chunks;       // column chunks of this sweep
  int item0;          // first work item of this sweep (items are [row tile fastest][column chunk])
  float* l_part;
  float* o_part;
  float* topv_part;
  int32_t* topi_part;
};
struct Sm100Params {
  int n_rows;
  int n_items;                // work items of the launch (all sub-sweeps); the CTA-pair kernel's persistent pairs walk this list
  const __nv_bfloat16* p16;   // [n_rows, D] probe rows (bf16), loaded straight into TMEM when P_TMEM
  const uint8_t* is_out;
  int32_t* kth_shared;        // [n_rows] shared hard-negative threshold (integer key), zeroed by the prep kernel
  // CTA-pair kernel: sweep position -> probe row, positives first and hard-negative-only ("outlier") rows last, and the number of
  // positives (device side).  Items whose rows are all at or beyond it run GEMM-1 and the top-k only.  NULL: identity, no such items.
  const int32_t* row_map;
  const int32_t* n_pos_dev;
  int32_t* done_flags;        // CTA-pair kernel, main sweep: [column chunk][row tile] == epoch once that item's top-k partial is in global memory
  int epoch;                  // (a later item of the same rows seeds its hard-negative lists from the finished items' partials)
  float a2, b2;       // p~ = 2^(a2 * z - b2)
  int k;
  int debug;   // bottleneck isolation BITMASK, only in FFC_SM100_DEBUG_BUILD builds; results are WRONG when any bit is set:
               // 1 = O-CTA skips TMA+MMA, 2 = epilogue skips tcgen05.ld/exp, 4 = S-CTA skips TMA+MMA,
               // 16 = no P~ hand-off (both CTAs free-run), 64 = no W TMA loads (MMAs run on whatever is in shared memory)
  SubSweep sub[MAX_SUB];
};

// host side (head_sm100.cu): cached tensor maps.  box = 64 features x box_rows rows (K-major, 128-byte swizzle); chunked3d: the same
// matrix as [D/64 chunks][rows][64] with one box = (64 features, box_rows rows, all chunks)
int sm100_get_map(Sm100Cache* c, const void* ptr, int64_t rows, int D, int box_rows, bool chunked3d, CUtensorMap* out);
// the one-CTA sweep for D <= 256 (head_sm100_1cta.cu)
int launch_sweeps_sm100_1cta(Sm100Cache* cache, const SweepArgs* sweeps, int n_sweeps, cudaStream_t s);
int sm100_1cta_tile_cols(int D);

}  // namespace ffc
