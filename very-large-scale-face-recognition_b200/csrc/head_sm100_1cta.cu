// One-CTA tcgen05 / TMEM / TMA sweep of the FFC head for feature widths D <= 256 (sm_100a).
//
// The CTA-pair kernel of head_sm100.cu exists because at D = 512 the fp32 gradient accumulator O[128 x 512] fills the 512 TMEM
// columns of an SM.  For D <= 256 everything fits ONE SM's tensor memory, and the pair only costs: every tile's p~ (32 KB) crosses
// DSMEM, and the exponentials of a tile -- 128 x 128 ex2 on a 16-per-clock MUFU pipe, 1 024 cycles, as long as the tile's GEMM-1 at
// D = 256 and twice as long at D = 128 -- run on one SM of the two while the other SM's MUFU pipe idles (measured round 1: 0.66 of the
// cuBLAS bf16 rate at D = 256, 0.37 at D = 128).  Here one CTA does both GEMMs of its tiles:
//
//   S[128 x BN]  = P . W_tile^T      tcgen05.mma, TS form: A = the probe tile P resident in TMEM (bf16 pairs, D/2 columns),
//                                    B = W K-chunks [BN rows x 64 features] streamed by TMA (K-major, 128-byte swizzle)
//   epilogue     8 warps (2 warpgroups = 2 S accumulators, tiles alternate): tcgen05.ld S, exclusions / SV transform,
//                p~ = 2^(a*cos - b), softmax denominator, hard-negative top-k, and p~ packed to bf16 is written with tcgen05.st
//                INTO THE COLUMNS S CAME FROM (the bf16 tile needs half of them): no shared-memory hand-off, no proxy fence
//   O[128 x D]  += P~ . W_tile        tcgen05.mma, TS form again: A = P~ in TMEM, B = the SAME shared-memory tile read MN-major
//
// BN = 128 queue rows per tile for D <= 128, 64 for D = 256 (TMEM: O D columns + 2 x BN for S / P~ + D/2 for P <= 512).  The tile
// ring holds whole tiles (a tile is read by GEMM-1 when it arrives and by GEMM-2 one epilogue later), 6 tiles of 32 KB at D = 128 / 256.
// MMAs of one CTA execute in issue order, so GEMM-1 of tile i+2 may overwrite the S / P~ buffer that GEMM-2 of tile i has just read
// without a barrier in between; the issue order is M1(0) M1(1) M2(0) M1(2) M2(1) ...: the tensor pipe works on GEMM-1 of the next
// tile while the epilogue of the current one runs.  Partial results (per column chunk: O, denominators, top-k) go to the same
// buffers as the pair kernel's, so prep / reduce / finalize do not care which kernel swept.
#include <cuda.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "sm100_ptx.cuh"

namespace ffc {
namespace one {

constexpr int BM = 128;            // probe rows per item
constexpr int KC = 64;             // bf16 elements per 128-byte swizzle row
constexpr int NEPI = 2;            // epilogue warpgroups == S / P~ accumulators
constexpr int NTHREADS = 128 + NEPI * 128;
constexpr int MAX_SLOTS = 8;       // tile slots of the ring

template <int D>
struct Shape {
  static constexpr int BN = D >= 256 ? 64 : 128;             // queue rows per tile
  static constexpr int NKC = D / KC;                          // K chunks of a tile
  static constexpr int CHUNK_BYTES = BN * KC * 2;
  static constexpr int TILE_BYTES = NKC * CHUNK_BYTES;
  static constexpr int SLOTS_RAW = (216 * 1024) / TILE_BYTES;
  static constexpr int SLOTS = SLOTS_RAW > MAX_SLOTS ? MAX_SLOTS : SLOTS_RAW;
  static constexpr int O_COL = 0, S_COL = D, P_COL = D + 2 * BN;      // tensor-memory columns
  static constexpr size_t SMEM = 1024 + (size_t)SLOTS * TILE_BYTES + 8 * 128 + 1024;   // barriers, ring, top-k scan staging, alignment slack
  static_assert(P_COL + D / 2 <= 512, "tensor memory budget");
  static_assert(SLOTS >= 3 && SMEM <= 227 * 1024, "shared memory budget");
};

struct Bars {
  uint64_t p_full;
  uint64_t w_full[MAX_SLOTS][4];
  uint64_t w_empty[MAX_SLOTS];
  uint64_t s_full[NEPI];
  uint64_t p_ready[NEPI];
  uint64_t o_full;
  uint32_t tmem_base;
  uint32_t pad;
};
static_assert(sizeof(Bars) <= 1024, "barrier block too large");

__device__ __forceinline__ void tc_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]),
      "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}

template <bool SV, int D>
__global__ void __launch_bounds__(NTHREADS, 1)
    ffc_head_sweep1_sm100_kernel(const __grid_constant__ CUtensorMap map_wa, const __grid_constant__ CUtensorMap map_wb,
                                 const __grid_constant__ CUtensorMap map_wc, const __grid_constant__ Sm100Params prm) {
  using Sh = Shape<D>;
  constexpr int BN = Sh::BN, NKC = Sh::NKC;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  Bars& bars = *reinterpret_cast<Bars*>(smem);
  unsigned char* sW = smem + 1024;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item_all = blockIdx.x;
  const int sidx = item_all >= prm.sub[2].item0 ? 2 : (item_all >= prm.sub[1].item0 ? 1 : 0);
  const SubSweep& sw = prm.sub[sidx];
  const CUtensorMap* map_w = sidx == 0 ? &map_wa : (sidx == 1 ? &map_wb : &map_wc);
  const int item = item_all - sw.item0;
  const int n_row_tiles = (prm.n_rows + BM - 1) / BM;
  const int rt = item % n_row_tiles, chunk = item / n_row_tiles;
  const int row0 = rt * BM;
  const int64_t n_cols = sw.n_cols_dev ? (int64_t)*sw.n_cols_dev : sw.n_cols;
  const int n_tiles_total = (int)((n_cols + BN - 1) / BN);
  const int t_begin = chunk * sw.tiles_per_chunk;
  int t_end = t_begin + sw.tiles_per_chunk;
  if (t_end > n_tiles_total) t_end = n_tiles_total;
  const int n_tiles = t_end > t_begin ? t_end - t_begin : 0;

  if (threadIdx.x == 0) {
    mbar_init(&bars.p_full, 4);
    for (int i = 0; i < MAX_SLOTS; ++i) {
      for (int kc = 0; kc < 4; ++kc) mbar_init(&bars.w_full[i][kc], 1);
      mbar_init(&bars.w_empty[i], 1);
    }
    for (int i = 0; i < NEPI; ++i) {
      mbar_init(&bars.s_full[i], 1);
      mbar_init(&bars.p_ready[i], 4);
    }
    mbar_init(&bars.o_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars.tmem_base)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars.tmem_base);

  if (warp == 0) {
    // ---- TMA producer: a tile = NKC boxes [BN rows x 64 features], each with its own full barrier (GEMM-1 starts on the first) ----
    int slot = 0;
    uint32_t ph = 0;
    for (int t = t_begin; t < t_end; ++t) {
      mbar_wait(&bars.w_empty[slot], ph ^ 1);
      if (elect_one()) {
#pragma unroll
        for (int kc = 0; kc < NKC; ++kc) {
          mbar_expect_tx(&bars.w_full[slot][kc], (uint32_t)Sh::CHUNK_BYTES);
          tma_load_2d(map_w, &bars.w_full[slot][kc], sW + slot * Sh::TILE_BYTES + kc * Sh::CHUNK_BYTES, kc * KC, t * BN);
        }
      }
      __syncwarp();
      if (++slot == Sh::SLOTS) {
        slot = 0;
        ph ^= 1;
      }
    }
  } else if (warp == 1) {
    // ---- MMA issue (converged warp, one elected lane): M1(0) M1(1) M2(0) M1(2) M2(1) ... ----
    if (n_tiles > 0) {
      constexpr uint32_t idesc1 = make_idesc(BM, BN, 0, 0);
      constexpr uint32_t idesc2 = make_idesc(BM, D, 0, 1);
      mbar_wait(&bars.p_full, 0);
      tc_fence_after();
      const uint64_t b1 = make_desc(smem_u32(sW), 16, 1024);                  // K-major tile chunks (GEMM-1)
      const uint64_t b2 = make_desc(smem_u32(sW), Sh::CHUNK_BYTES, 1024);      // the same bytes MN-major (GEMM-2): 64-feature atoms one chunk apart
      const uint32_t tmem_o = tmem_base + (uint32_t)Sh::O_COL;
      int slot1 = 0;        // ring slot / phase of the next GEMM-1 tile
      uint32_t ph1 = 0;
      auto issue_m1 = [&](int t) {
        const uint32_t tmem_s = tmem_base + (uint32_t)(Sh::S_COL + (t & 1) * BN);
#pragma unroll
        for (int kc = 0; kc < NKC; ++kc) {
          mbar_wait(&bars.w_full[slot1][kc], ph1);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t bd = b1 + (uint64_t)((slot1 * Sh::TILE_BYTES + kc * Sh::CHUNK_BYTES) >> 4);
            const uint32_t ta = tmem_base + (uint32_t)(Sh::P_COL + kc * (KC / 2));
#pragma unroll
            for (int k = 0; k < KC / 16; ++k) tc_mma_ts(tmem_s, ta + (uint32_t)(8 * k), bd + (uint64_t)(2 * k), idesc1, (kc | k) ? 1u : 0u);
            if (kc == NKC - 1) tc_commit(&bars.s_full[t & 1]);
          }
          __syncwarp();
        }
        if (++slot1 == Sh::SLOTS) {
          slot1 = 0;
          ph1 ^= 1;
        }
      };
      issue_m1(0);
      int slot2 = 0;
      for (int i = 0; i < n_tiles; ++i) {
        if (i + 1 < n_tiles) issue_m1(i + 1);
        mbar_wait(&bars.p_ready[i & 1], (uint32_t)(i >> 1) & 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t ta = tmem_base + (uint32_t)(Sh::S_COL + (i & 1) * BN);       // P~ sits in the first BN/2 columns of its S buffer
          const uint64_t bs = b2 + (uint64_t)((slot2 * Sh::TILE_BYTES) >> 4);
#pragma unroll
          for (int k16 = 0; k16 < BN / 16; ++k16)
            tc_mma_ts(tmem_o, ta + (uint32_t)(8 * k16), bs + (uint64_t)(k16 * ((16 * 128) >> 4)), idesc2, (i | k16) ? 1u : 0u);
          tc_commit(&bars.w_empty[slot2]);        // the tile's slot is free once GEMM-2 has read it
          if (i == n_tiles - 1) tc_commit(&bars.o_full);
        }
        __syncwarp();
        if (++slot2 == Sh::SLOTS) slot2 = 0;
      }
    }
  } else if (warp >= 4) {
    // ---- epilogue: warpgroup g takes the tiles of parity g (S / P~ buffer g) ----
    const int g = (warp - 4) >> 2;
    const int q4 = warp & 3;                    // TMEM lane quarter
    const int r_local = q4 * 32 + lane;
    const int row = row0 + r_local;
    const bool row_ok = row < prm.n_rows;
    const int32_t tcol = (row_ok && sw.tcol) ? sw.tcol[row] : -1;
    const bool outl = row_ok && prm.is_out && prm.is_out[row];
    const bool warp_out = __any_sync(0xffffffffu, outl);
    float thr = INFINITY;
    if (SV && row_ok && sw.thr) thr = sw.thr[row];
    const float a2 = prm.a2, b2 = prm.b2;
    const int k = prm.k;
    float lsum = 0.f;
    int tk[KMAX], tc[KMAX];
#pragma unroll
    for (int q = 0; q < KMAX; ++q) {
      tk[q] = 0;
      tc[q] = -1;
    }
    int kth = 0;
    uint32_t* scan_stage = reinterpret_cast<uint32_t*>(sW + Sh::SLOTS * Sh::TILE_BYTES) + (warp - 4) * 32;   // 128 bytes per epilogue warp
    int32_t* kshare = (sidx == 0 && outl && prm.kth_shared) ? prm.kth_shared + row : nullptr;      // threshold shared by the column chunks of a row (see head_sm100.cu)
    int kfloor = 0, kpub = 0;
    float pthr = __uint_as_float(__float_as_uint(ex2f(-b2)) & 0xffff0000u);
    const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16);
    if (g == 0 && n_tiles > 0) {
      // probe tile -> TMEM (the A operand of every GEMM-1 of this item): thread = row, 32 columns (64 bf16) per store
      const uint4* src = reinterpret_cast<const uint4*>(prm.p16 + (int64_t)(row_ok ? row : 0) * D);
#pragma unroll 1
      for (int c0 = 0; c0 < D / 2; c0 += 32) {
        uint32_t v[32];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const uint4 t = row_ok ? __ldg(src + c0 / 4 + q) : make_uint4(0u, 0u, 0u, 0u);
          v[4 * q] = t.x;
          v[4 * q + 1] = t.y;
          v[4 * q + 2] = t.z;
          v[4 * q + 3] = t.w;
        }
        tc_st32(lane_base + (uint32_t)(Sh::P_COL + c0), v);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.p_full);
    }
    uint32_t use = 0;
    for (int i = g; i < n_tiles; i += NEPI, ++use) {
      const int j0 = (t_begin + i) * BN;
      uint32_t cmw[BN / 32];
#pragma unroll
      for (int cc = 0; cc < BN / 32; ++cc) cmw[cc] = (sw.cmask && (int64_t)j0 + cc * 32 < n_cols) ? __ldg(sw.cmask + (j0 >> 5) + cc) : 0u;
      int kshared = 0;
      if (kshare) kshared = __ldcg(kshare);
      mbar_wait(&bars.s_full[g], use & 1);
      tc_fence_after();
      const uint32_t tmem_s = lane_base + (uint32_t)(Sh::S_COL + g * BN);
      kfloor = max(kfloor, kshared);
      kth = max(kth, kfloor);
      if (!SV && warp_out) pthr = __uint_as_float(__float_as_uint(ex2f(fmaf(__int_as_float(kth & (int)TOPK_VAL_MASK), a2, -b2))) & 0xffff0000u);
      float l0 = 0.f, l1 = 0.f;
#pragma unroll 1
      for (int cc = 0; cc < BN / 32; ++cc) {
        uint32_t v[32];
        tc_ld32(tmem_s + cc * 32, v);
        const int col0 = j0 + cc * 32;
        uint32_t excl = cmw[0];
#pragma unroll
        for (int q = 1; q < BN / 32; ++q)
          if (cc == q) excl = cmw[q];
        const int trel = tcol - col0;
        if ((unsigned)trel < 32u) excl |= 1u << trel;
        if ((int64_t)col0 + 32 > n_cols) {
          const int nv = (int)(n_cols - col0);
          excl |= nv <= 0 ? 0xffffffffu : (0xffffffffu << nv);
        }
        const bool slow = __any_sync(0xffffffffu, excl != 0u);
        uint32_t pk[16];
#pragma unroll
        for (int c = 0; c < 32; c += 2) {
          const float x0 = __uint_as_float(v[c]), x1 = __uint_as_float(v[c + 1]);
          float p0, p1, g0, g1;
          if (SV) {
            const bool m0 = x0 > thr, m1 = x1 > thr;
            p0 = ex2f(fmaf(m0 ? fmaf(SV_T, x0, SV_T - 1.f) : x0, a2, -b2));
            p1 = ex2f(fmaf(m1 ? fmaf(SV_T, x1, SV_T - 1.f) : x1, a2, -b2));
            g0 = m0 ? p0 * SV_T : p0;
            g1 = m1 ? p1 * SV_T : p1;
          } else {
            p0 = g0 = ex2f(fmaf(x0, a2, -b2));
            p1 = g1 = ex2f(fmaf(x1, a2, -b2));
          }
          if (slow) {
            if ((excl >> c) & 1u) p0 = g0 = 0.f;
            if ((excl >> (c + 1)) & 1u) p1 = g1 = 0.f;
          }
          l0 += p0;
          l1 += p1;
          pk[c >> 1] = pack_bf16(g0, g1);
        }
        // ---- hard-negative top-k on the raw cosines of outlier rows (as in head_sm100.cu) ----
        if (SV) {
          if (warp_out) {
            topk_scan16<0, 32>(v, excl & 0xffffu, col0, outl, k, tk, tc, kth, kfloor);
            topk_scan16<16, 32>(v, excl >> 16, col0 + 16, outl, k, tk, tc, kth, kfloor);
          }
        } else if (warp_out) {
          uint32_t m = pk[0];
#pragma unroll
          for (int q = 1; q < 16; ++q) m = max_bf16x2(m, pk[q]);
          const float mf = fmaxf(__uint_as_float(m << 16), __uint_as_float(m & 0xffff0000u));
          unsigned cand = __ballot_sync(0xffffffffu, outl && mf >= pthr);
          if (cand) {
            if (__popc(cand) > 4) {
              topk_scan16<0, 32>(v, excl & 0xffffu, col0, outl, k, tk, tc, kth, kfloor);
              topk_scan16<16, 32>(v, excl >> 16, col0 + 16, outl, k, tk, tc, kth, kfloor);
              cand = 0u;
            }
            while (cand) {
              const int L = __ffs(cand) - 1;
              cand &= cand - 1;
              if (lane == L) {
#pragma unroll
                for (int q = 0; q < 8; ++q) *reinterpret_cast<uint4*>(scan_stage + 4 * q) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
              }
              __syncwarp();
              const uint32_t exclL = __shfl_sync(0xffffffffu, excl, L);
              const int key = ((exclL >> lane) & 1u) ? 0 : (int)((scan_stage[lane] & TOPK_VAL_MASK) | (uint32_t)lane);
              const int kthL = __shfl_sync(0xffffffffu, kth, L);
              unsigned hits = __ballot_sync(0xffffffffu, key > kthL);
              while (hits) {
                const int c = __ffs(hits) - 1;
                hits &= hits - 1;
                const int kc = __shfl_sync(0xffffffffu, key, c);
                if (lane == L && kc > kth) {
                  topk_insert_key(kc, col0, k, tk, tc);
#pragma unroll
                  for (int r = 0; r < KMAX; ++r)
                    if (r == k - 1) kth = max(tk[r], kfloor);
                }
              }
              __syncwarp();
            }
            pthr = __uint_as_float(__float_as_uint(ex2f(fmaf(__int_as_float(kth & (int)TOPK_VAL_MASK), a2, -b2))) & 0xffff0000u);
          }
        }
        // P~[row][cc*32 .. +32) as 16 packed columns over the first half of the S columns just read (the writes trail the reads:
        // chunk cc lands in columns [16 cc, 16 cc + 16), all inside S chunks <= cc)
        tc_st16(tmem_s + cc * 16, pk);
      }
      lsum += l0 + l1;
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.p_ready[g]);
      if (kshare) {
        int kown = 0;
#pragma unroll
        for (int r = 0; r < KMAX; ++r)
          if (r == k - 1) kown = tk[r];
        if (kown > kpub) {
          atomicMax(kshare, kown);
          kpub = kown;
        }
      }
    }
    // ---- item end: O write-out (warpgroup g: half of the features), then the two warpgroups' scalars are merged through the idle ring ----
    if (n_tiles > 0) {
      mbar_wait(&bars.o_full, 0);      // every MMA of the item has completed: O is final, the ring is idle
      tc_fence_after();
    }
    {
      constexpr int half = D / 2;
      // each warp transposes its 32 x 32 block through 4.5 KB of the idle ring (beyond the 16 KB the scalar merge below uses), so
      // that a store instruction covers 4 rows x 128 contiguous bytes instead of 32 rows x 16 bytes (see head_sm100.cu)
      float* stg = reinterpret_cast<float*>(sW + 16384) + (warp - 4) * (32 * 36);
      float* dst0 = sw.o_part + ((int64_t)chunk * prm.n_rows + row0 + q4 * 32) * D + g * half;
#pragma unroll 1
      for (int c0 = 0; c0 < half; c0 += 32) {
        uint32_t v[32];
        if (n_tiles > 0) {
          tc_ld32(lane_base + (uint32_t)(Sh::O_COL + g * half + c0), v);
        } else {
#pragma unroll
          for (int c = 0; c < 32; ++c) v[c] = 0u;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) *reinterpret_cast<uint4*>(stg + lane * 36 + 4 * q) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int r = it * 4 + (lane >> 3), c = (lane & 7) * 4;
          const uint4 x = *reinterpret_cast<const uint4*>(stg + r * 36 + c);
          if (row0 + q4 * 32 + r < prm.n_rows) *reinterpret_cast<uint4*>(dst0 + (int64_t)r * D + c0 + c) = x;
        }
        __syncwarp();
      }
      tc_fence_before();
    }
    float* stage_v = reinterpret_cast<float*>(sW);                             // [128][KMAX]
    int32_t* stage_i = reinterpret_cast<int32_t*>(sW + BM * KMAX * 4);         // [128][KMAX]
    float* stage_l = reinterpret_cast<float*>(sW + 2 * BM * KMAX * 4);         // [128]
    float tv[KMAX];
    int32_t ti[KMAX];
#pragma unroll
    for (int q = 0; q < KMAX; ++q) {
      const bool live = tk[q] > 0;
      tv[q] = live ? __int_as_float(tk[q] & (int)TOPK_VAL_MASK) : -INFINITY;
      ti[q] = live ? tc[q] + (tk[q] & 31) : -1;
    }
    if (g == 1) {
      stage_l[r_local] = lsum;
#pragma unroll
      for (int q = 0; q < KMAX; ++q) {
        stage_v[r_local * KMAX + q] = tv[q];
        stage_i[r_local * KMAX + q] = ti[q];
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (g == 0 && row_ok) {
      float kthv = -INFINITY;
#pragma unroll
      for (int q = 0; q < KMAX; ++q)
        if (q == k - 1) kthv = tv[q];
      lsum += stage_l[r_local];
      if (outl) {
#pragma unroll 1
        for (int q = 0; q < k; ++q) {
          const float x = stage_v[r_local * KMAX + q];
          if (x > kthv) {
            topk_insert<KMAX>(tv, ti, k, x, stage_i[r_local * KMAX + q]);
#pragma unroll
            for (int qq = 0; qq < KMAX; ++qq)
              if (qq == k - 1) kthv = tv[qq];
          }
        }
      }
      const int64_t pr = (int64_t)chunk * prm.n_rows + row;
      sw.l_part[pr] = lsum;
#pragma unroll
      for (int q = 0; q < KMAX; ++q) {
        if (q < k) {
          sw.topv_part[pr * k + q] = tv[q];
          sw.topi_part[pr * k + q] = ti[q];
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
}

template <bool SV, int D>
static int launch_one(const CUtensorMap* maps, const Sm100Params& p, int n_items, cudaStream_t s) {
  static bool attr_set = false;
  auto kern = ffc_head_sweep1_sm100_kernel<SV, D>;
  constexpr size_t smem = Shape<D>::SMEM;
  if (!attr_set) {
    FFC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  kern<<<dim3(n_items), dim3(NTHREADS), smem, s>>>(maps[0], maps[1], maps[2], p);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

}  // namespace one

int sm100_1cta_tile_cols(int D) { return D >= 256 ? 64 : 128; }

// as launch_sweeps_sm100 (head_sm100.cu): `sweeps[0 .. n_sweeps)` share P, n_rows, D, is_out, scale, fixed_max, sv and k
int launch_sweeps_sm100_1cta(Sm100Cache* cache, const SweepArgs* sweeps, int n_sweeps, cudaStream_t s) {
  FFC_REQUIRE(n_sweeps >= 1 && n_sweeps <= MAX_SUB, "tcgen05 sweep: %d sweeps per launch (1..%d)", n_sweeps, MAX_SUB);
  const SweepArgs& a = sweeps[0];
  FFC_REQUIRE(a.D == 64 || a.D == 128 || a.D == 256, "one-CTA tcgen05 sweep: D=%d must be 64, 128 or 256", a.D);
  FFC_REQUIRE(a.P_bf16, "tcgen05 sweep: bf16 operands missing");
  FFC_REQUIRE(!a.W2_bf16, "one-CTA tcgen05 sweep: both GEMMs read the same tile (W2 needs the CTA-pair kernel)");
  const int BN = sm100_1cta_tile_cols(a.D);
  CUtensorMap maps[MAX_SUB];
  Sm100Params p;
  memset(&p, 0, sizeof(p));
  p.n_rows = a.n_rows;
  p.p16 = a.P_bf16;
  p.is_out = a.is_out;
  p.kth_shared = a.kth_shared;
  p.a2 = a.scale * LOG2E;
  p.b2 = a.fixed_max * LOG2E;
  p.k = a.k;
  const int row_tiles = (a.n_rows + one::BM - 1) / one::BM;
  int n_items = 0, rc;
  for (int i = 0; i < MAX_SUB; ++i) {
    SubSweep& sb = p.sub[i];
    if (i >= n_sweeps) {
      sb.item0 = 0x7fffffff;
      maps[i] = maps[0];
      continue;
    }
    const SweepArgs& w = sweeps[i];
    FFC_REQUIRE(w.W_bf16 && w.n_rows == a.n_rows && w.D == a.D && w.P_bf16 == a.P_bf16 && w.sv == a.sv && w.k == a.k && w.n_chunks >= 1,
                "tcgen05 sweep: sweep %d does not share the probe rows / shape of sweep 0", i);
    if ((rc = sm100_get_map(cache, w.W_bf16, w.n_cols, w.D, BN, false, &maps[i]))) return rc;
    sb.n_cols = w.n_cols;
    sb.n_cols_dev = w.n_cols_dev;
    sb.tcol = w.tcol;
    sb.cmask = w.cmask;
    sb.thr = w.thr;
    const int64_t n_tiles = std::max<int64_t>(1, ceil_div64(w.n_cols, BN));
    sb.tiles_per_chunk = (int)ceil_div64(n_tiles, w.n_chunks);
    sb.item0 = n_items;
    sb.l_part = w.l_part;
    sb.o_part = w.o_part;
    sb.topv_part = w.topv_part;
    sb.topi_part = w.topi_part;
    n_items += row_tiles * w.n_chunks;
  }
#define FFC_SWEEP1_CASE(DV) \
  case DV:                  \
    return a.sv ? one::launch_one<true, DV>(maps, p, n_items, s) : one::launch_one<false, DV>(maps, p, n_items, s);
  switch (a.D) {
    FFC_SWEEP1_CASE(64)
    FFC_SWEEP1_CASE(128)
    FFC_SWEEP1_CASE(256)
  }
#undef FFC_SWEEP1_CASE
  return FFC_ERR_INVALID;
}

}  // namespace ffc
