// tcgen05 / TMEM / TMA sweep of the FFC head for sm_100a (the hot kernel).
//
// One work item = (128 probe rows) x (a contiguous range of 128-row queue tiles), processed by a
// CLUSTER OF TWO CTAs with different roles, because at D = 512 the fp32 gradient accumulator
// O[128 x 512] alone fills the 512 TMEM columns of one SM:
//
//   CTA rank 0, "S-CTA":  S = P . W_tile^T        (tcgen05.mma TS form, M=128 N=128 K=D: A = the probe tile P resident in
//                          TMEM, B = W K-chunks streamed by TMA through a 12-stage ring);  12 epilogue warps read S from
//                          TMEM, apply exclusions / SV transform, p~ = 2^(a*cos - b), accumulate the softmax denominator and
//                          the running top-k, and store p~ as bf16 straight into the peer CTA's shared memory (st.async) in
//                          the interleaved K-major layout the second GEMM reads (512 contiguous bytes per warp store).
//   CTA rank 1, "O-CTA":  O += P~ . W_tile          (tcgen05.mma SS form, M=128 N<=256 per instruction, K=128 queue rows per
//                          tile, A = P~ from smem, B = the same W tile, one 3-D TMA box per stage, read MN-major);  O stays
//                          in TMEM for the whole item and is written once.
//
// Executed tensor FLOPs == algorithmic FLOPs (4 * rows * cols * D): no recompute, no B x Q logits.  One launch carries the
// main sweep and the two side sweeps of a pass.  Every MMA / TMA warp runs converged with one elected lane issuing.
// Synchronisation is all mbarriers: TMA -> MMA (full/empty rings), MMA -> epilogue (tcgen05.commit, one barrier per
// epilogue warpgroup), epilogue -> peer hand-off warp (st.async complete_tx on the peer's mbarrier) -> peer MMA,
// peer MMA -> epilogue (multicast tcgen05.commit).
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "head_internal.cuh"
#include "sm100_ptx.cuh"

namespace ffc {

constexpr int BM = 128;            // probe rows per item
constexpr int BN = 128;            // queue rows per tile
constexpr int KC = 64;             // bf16 elements per 128-byte swizzle row
#ifndef FFC_NS1
#define FFC_NS1 12
#endif
#ifndef FFC_JB
#define FFC_JB 32
#endif
constexpr int NS1 = FFC_NS1;       // S-CTA W K-chunk stages (16 KB each)
constexpr int NSB = 2;             // S accumulators in the S-CTA's TMEM (128 columns each): S0 S1 | P (D/2 columns at 256)
constexpr int P_TMEM_COL = 256;
constexpr int NPB = 3;             // P~ buffers in the O-CTA's shared memory
constexpr int JB = FFC_JB;         // queue rows per O-CTA W stage
constexpr int NEPI = 3;             // epilogue warpgroups in the S-CTA (tiles are dealt round-robin)
constexpr int NTHREADS = 128 + NEPI * 128;   // 4 control warps + 12 epilogue warps
constexpr int CHUNK1_BYTES = BN * KC * 2;   // 16384

// ---- shared memory map (same for both roles; 1024-byte aligned base) ----
// [0, 1024)                 barriers, tmem base
// S-CTA: [1024, ...)        NS1 x 16 KB W chunk ring (K-major SW128), 12 x 128 B top-k scan staging, then the end-of-item staging of the
//                           epilogue warpgroups' per-row partials ([2][128] denominators, [2][128][KMAX] top-k values and columns)
// O-CTA: [1024, +96K)       P~ buffers 3 x 32 KB (interleaved K-major), then NS2 x (D/64 * 4 KB) W stage ring
// ---- tensor memory (512 columns per SM) ----
// S-CTA: [0, 256) two S accumulators, [256, 256 + D/2) the probe tile P as packed bf16 pairs (lane = row)
// O-CTA: [0, D) the fp32 gradient accumulator O
constexpr int OFF_DATA = 1024;
constexpr int PT_BYTES = BM * BN * 2;       // 32768 per P~ buffer
constexpr int SCAN_STAGE_BYTES = NEPI * 4 * 128;
constexpr int ITEM_STAGE_BYTES = (NEPI - 1) * BM * (4 + 8 * KMAX);

struct Bars {   // all in the first 1024 bytes
  uint64_t p_full;                 // the item's probe tile is in TMEM (12 epilogue warps arrive, once per item)
  uint64_t w_full[NS1], w_empty[NS1];
  uint64_t s_full[NEPI];           // one per epilogue warpgroup (NOT per S buffer): each is waited by one warpgroup, in order
  uint64_t s_empty[NSB];
  uint64_t pt_empty[NPB];          // S-CTA side: P~ buffer b may be overwritten (signalled by the peer's tcgen05.commit, or by its O
                                   // write-out warps for the buffer they used as staging)
  uint64_t w2_full[8], w2_empty[8];
  uint64_t pt_full[NPB];           // O-CTA side: P~ buffer b is complete (st.async complete_tx, 32 KB per tile)
  uint64_t pt_ready[NPB];          // O-CTA side: ... and the proxy fence that lets tcgen05.mma read it has been executed
  uint64_t o_full;                 // O-CTA: every tcgen05.mma of the item has completed (O may be read)
  uint64_t o_empty;                // O-CTA: the item's O has been read out of TMEM (the next item may overwrite it)
  uint32_t tmem_base;
  uint32_t pad;
};
static_assert(sizeof(Bars) <= 1024, "barrier block too large");

// Byte offset of the 16-byte piece `piece` (= 8 consecutive queue columns, 0..15) of row `r` inside one 32 KB P~ buffer:
// the interleaved (SWIZZLE_NONE) K-major layout, 8x16-byte core matrices with the 128 rows of one piece contiguous
// (2 KB).  The 32 lanes of a warp (32 consecutive rows) therefore write 512 contiguous bytes per store instruction --
// coalesced DSMEM traffic (hand-off alone: 0.80 ms per sweep, against 1.47 ms for 128-byte-strided SWIZZLE_128B rows).
__device__ __forceinline__ uint32_t pt_offset(uint32_t piece, uint32_t r) { return piece * (uint32_t)(BM * 16) + r * 16u; }

#ifndef FFC_SM100_DEBUG_BUILD
#define FFC_SM100_DEBUG_BUILD 0     // 1: honour Sm100Params::debug (bottleneck isolation, see tools/sweep_modes.py)
#endif

#if FFC_SM100_DEBUG_BUILD
// per-CTA phase stamps of the last launch: [cta][0..5] = clock64 at start / set-up done / first MMA loop start / last MMA loop end /
// role work done / after the final cluster sync; [6], [7] = globaltimer (ns) at start / end
__device__ long long g_sweep_stamps[1024][8];
#define FFC_STAMP(slot)                                                                    \
  do {                                                                                     \
    if (blockIdx.x < 1024) g_sweep_stamps[blockIdx.x][slot] = clock64();                   \
  } while (0)
#define FFC_STAMP_NS(slot)                                                                 \
  do {                                                                                     \
    long long t_;                                                                          \
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                 \
    if (blockIdx.x < 1024) g_sweep_stamps[blockIdx.x][slot] = t_;                          \
  } while (0)
// per-CTA cycle sums: [0] MMA warp waiting for its accumulator / P~ buffer, [1] MMA warp waiting for W (TMA), [2] MMA warp
// issuing, [3] epilogue warp 4 waiting for S, [4] epilogue warp 4 waiting for a free P~ buffer, [5] epilogue warp 4 working,
// [6] TMA producer waiting for a free stage, [7] S-CTA: top-k scan triggers; O-CTA: MMA warp between two items (O read-out)
__device__ long long g_sweep_prof[1024][8];
#define FFC_PROF_DECL(name) long long name = 0
#define FFC_PROF_T(var) const long long var = clock64()
#define FFC_PROF_ADD(acc, t0, t1) acc += (t1) - (t0)
#define FFC_PROF_STORE(slot, acc)                                                          \
  do {                                                                                     \
    if (blockIdx.x < 1024) g_sweep_prof[blockIdx.x][slot] = (acc);                         \
  } while (0)
#else
#define FFC_PROF_DECL(name) do {} while (0)
#define FFC_PROF_T(var) do {} while (0)
#define FFC_PROF_ADD(acc, t0, t1) do {} while (0)
#define FFC_PROF_STORE(slot, acc) do {} while (0)
#define FFC_STAMP(slot) do {} while (0)
#define FFC_STAMP_NS(slot) do {} while (0)
#endif

template <int D>
struct SweepShape {
  static constexpr int NKC = D / KC;                         // 64-column K chunks of the feature dim
  static constexpr int STAGE2_BYTES = NKC * JB * KC * 2;     // O-CTA stage: JB queue rows x D
  static constexpr int NS2_RAW = (225 * 1024 - NPB * PT_BYTES) / STAGE2_BYTES;
  static constexpr int NS2 = NS2_RAW > 8 ? 8 : (NS2_RAW < 2 ? 2 : NS2_RAW);
  static constexpr int N2 = D < 256 ? D : 256;               // GEMM-2 instruction N
  static constexpr int NHALF = (D + 255) / 256;              // GEMM-2 instructions per K step
  static constexpr size_t SMEM_S = OFF_DATA + (size_t)NS1 * CHUNK1_BYTES + SCAN_STAGE_BYTES + ITEM_STAGE_BYTES;
  static constexpr size_t SMEM_O = OFF_DATA + NPB * (size_t)PT_BYTES + (size_t)NS2 * STAGE2_BYTES;
  static constexpr size_t SMEM = (SMEM_S > SMEM_O ? SMEM_S : SMEM_O) + 1024;   // slack for the 1024-byte alignment of the base
  static_assert(SMEM <= 227 * 1024, "shared memory budget exceeded");
};

// A work item = (sub-sweep, row tile, column chunk).  Items are numbered [sub-sweep][column chunk][row tile fastest]; a CTA pair
// works through items pair, pair + n_pairs, ... (every role of both CTAs decodes the same sequence on its own).
struct Item {
  int sidx, chunk, row0, t_begin, n_tiles;
  int64_t n_cols;
  bool all_out;      // every probe row of the item is a hard-negative-only row (see Sm100Params::row_map): no softmax term, no GEMM-2
};
__device__ __forceinline__ Item decode_item(const Sm100Params& prm, int item_all) {
  Item it;
  it.sidx = item_all >= prm.sub[2].item0 ? 2 : (item_all >= prm.sub[1].item0 ? 1 : 0);
  const SubSweep& sw = prm.sub[it.sidx];
  const int item = item_all - sw.item0;
  const int n_row_tiles = (prm.n_rows + BM - 1) / BM;
  it.chunk = item / n_row_tiles;
  it.row0 = (item - it.chunk * n_row_tiles) * BM;
  it.n_cols = sw.n_cols_dev ? (int64_t)*sw.n_cols_dev : sw.n_cols;
  const int n_tiles_total = (int)((it.n_cols + BN - 1) / BN);
  it.t_begin = it.chunk * sw.tiles_per_chunk;
  int t_end = it.t_begin + sw.tiles_per_chunk;
  if (t_end > n_tiles_total) t_end = n_tiles_total;
  it.n_tiles = t_end > it.t_begin ? t_end - it.t_begin : 0;
  it.all_out = prm.n_pos_dev != nullptr && it.row0 >= *prm.n_pos_dev;
  return it;
}

// DQ_SV: the SV queue-gradient sweep (ffc_head_dqueue on an SV head, roles swapped: the columns are the probe rows).  P~ is then the
// combined weight sum_l a_l,j p~_l,ij h'_l,ij of both losses, from per-column thresholds and coefficients (Sm100Params::dq_col), and
// GEMM-2 accumulates the raw probe rows.
template <bool SV, int D, bool DQ_SV = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
    ffc_head_sweep_sm100_kernel(const __grid_constant__ CUtensorMap map_p, const __grid_constant__ CUtensorMap map_w1a,
                                const __grid_constant__ CUtensorMap map_w2a, const __grid_constant__ CUtensorMap map_w1b,
                                const __grid_constant__ CUtensorMap map_w2b, const __grid_constant__ CUtensorMap map_w1c,
                                const __grid_constant__ CUtensorMap map_w2c, const __grid_constant__ Sm100Params prm) {
  using Sh = SweepShape<D>;
  constexpr int NKC = Sh::NKC;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // SWIZZLE_128B operands need a 1024-byte aligned base; both CTAs of the pair compute the same offset
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  Bars& bars = *reinterpret_cast<Bars*>(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  // Item loop: pair p works through items p, p + n_pairs, ...  The default launch has one pair per item (the loop runs once and the
  // hardware deals the items to the SMs); a persistent launch (see persistent_grid) has fewer pairs than items.  Barriers, tensor
  // memory and the pipeline rings are set up once and their phases run on across items, so between two items only the data
  // dependencies remain: the S-CTA reloads P once the item's last GEMM-1 has completed, the O-CTA's next item starts once O has been
  // read out of TMEM -- while the W rings are already being refilled and the S-CTA works two P~ tiles ahead.
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int n_items = prm.n_items;
  const int dbg = FFC_SM100_DEBUG_BUILD ? prm.debug : 0;
  const bool dbg_noO = (dbg & 1) != 0, dbg_noEpi = (dbg & 2) != 0, dbg_noS = (dbg & 4) != 0, dbg_noHand = (dbg & 16) != 0, dbg_noTma = (dbg & 64) != 0;
  (void)map_p;

  if (threadIdx.x == 0) {
    FFC_STAMP(0);
    FFC_STAMP_NS(6);
  }
  unsigned char* sW1 = smem + OFF_DATA;                        // S-CTA (P lives in TMEM)
  unsigned char* sPt = smem + OFF_DATA;                        // O-CTA
  unsigned char* sW2 = sPt + NPB * PT_BYTES;                   // O-CTA

  if (threadIdx.x == 0) {
    mbar_init(&bars.p_full, 4 * NEPI);
    for (int i = 0; i < NS1; ++i) {
      mbar_init(&bars.w_full[i], 1);
      mbar_init(&bars.w_empty[i], 1);
    }
    for (int i = 0; i < NEPI; ++i) mbar_init(&bars.s_full[i], 1);
    for (int i = 0; i < NSB; ++i) mbar_init(&bars.s_empty[i], 4);
    for (int i = 0; i < NPB; ++i) {
      mbar_init(&bars.pt_empty[i], 1);
      mbar_init(&bars.pt_full[i], 1);
      mbar_init(&bars.pt_ready[i], 1);
    }
    for (int i = 0; i < 8; ++i) {
      mbar_init(&bars.w2_full[i], 1);
      mbar_init(&bars.w2_empty[i], 1);
    }
    mbar_init(&bars.o_full, 1);
    mbar_init(&bars.o_empty, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    // S-CTA: NSB x 128 columns of S + P; O-CTA: D columns of O (power of two >= 32)
    const uint32_t ncols = rank == 0 ? 512u : (uint32_t)(D < 32 ? 32 : D);
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars.tmem_base)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars.tmem_base);
  if (threadIdx.x == 0) FFC_STAMP(1);
  if (rank == 0) {
    // =========================================== S-CTA ===========================================
    if (warp == 0) {
      // ---- TMA producer (converged warp, one elected lane issues); runs ahead into the next item as far as the ring allows ----
      int stage = 0;
      uint32_t ph = 0;
      FFC_PROF_DECL(prof_tma);
      for (int ia = pair; ia < n_items; ia += n_pairs) {
        const Item it = decode_item(prm, ia);
        if (it.n_tiles == 0 || dbg_noS || dbg_noTma) continue;
        const CUtensorMap* map_w1 = it.sidx == 0 ? &map_w1a : (it.sidx == 1 ? &map_w1b : &map_w1c);
        for (int t = it.t_begin; t < it.t_begin + it.n_tiles; ++t) {
#pragma unroll
          for (int kc = 0; kc < NKC; ++kc) {
            FFC_PROF_T(q0);
            mbar_wait(&bars.w_empty[stage], ph ^ 1);
            FFC_PROF_T(q1);
            FFC_PROF_ADD(prof_tma, q0, q1);
            if (elect_one()) {
              mbar_expect_tx(&bars.w_full[stage], CHUNK1_BYTES);
              tma_load_2d(map_w1, &bars.w_full[stage], sW1 + stage * CHUNK1_BYTES, kc * KC, t * BN);
            }
            __syncwarp();
            if (++stage == NS1) {
              stage = 0;
              ph ^= 1;
            }
          }
        }
      }
      if (lane == 0) FFC_PROF_STORE(6, prof_tma);
    } else if (warp == 1) {
      // ---- GEMM-1 issue: S[128 x 128] = P[128 x D] . W_tile[128 x D]^T, 4 x (K = 16) per 64-column chunk ----
      constexpr uint32_t idesc = make_idesc(BM, BN, 0, 0);
      const uint64_t b0 = make_desc(smem_u32(sW1), 16, 1024);
      int stage = 0;
      uint32_t ph = 0;
      uint32_t gi = 0;      // tiles issued by this CTA so far (all items): tile gi uses S buffer gi % NSB and epilogue warpgroup gi % NEPI
      int wg = 0;
      uint32_t ni = 0;      // items with tiles so far
      bool stamped = false;
      FFC_PROF_DECL(prof_a);
      FFC_PROF_DECL(prof_b);
      FFC_PROF_DECL(prof_c);
      for (int ia = pair; ia < n_items; ia += n_pairs) {
        const Item it = decode_item(prm, ia);
        if (it.n_tiles == 0) continue;
        if (!dbg_noS) mbar_wait(&bars.p_full, ni & 1);       // the item's probe tile is in TMEM
        tc_fence_after();
        if (!stamped && lane == 0) FFC_STAMP(2);
        stamped = true;
        for (int i = 0; i < it.n_tiles; ++i, ++gi, wg = (wg + 1 == NEPI ? 0 : wg + 1)) {
          const int sb = (int)(gi & (NSB - 1));
          FFC_PROF_T(q0);
          mbar_wait(&bars.s_empty[sb], ((gi / NSB) & 1) ^ 1);
          tc_fence_after();
          FFC_PROF_T(q1);
          FFC_PROF_ADD(prof_a, q0, q1);
          if (dbg_noS) {
            if (elect_one()) mbar_arrive(&bars.s_full[wg]);
            __syncwarp();
            continue;
          }
          const uint32_t tmem_s = tmem_base + (uint32_t)(sb * BN);
#pragma unroll
          for (int kc = 0; kc < NKC; ++kc) {
            FFC_PROF_T(q2);
            if (!dbg_noTma) {
              mbar_wait(&bars.w_full[stage], ph);
              tc_fence_after();
            }
            FFC_PROF_T(q3);
            FFC_PROF_ADD(prof_b, q2, q3);
            if (elect_one()) {
              const uint64_t bd = b0 + (uint64_t)(stage * (CHUNK1_BYTES >> 4));
              // A = P[128 x 16] from TMEM: lane = probe row, 8 columns (two bf16 per column) per K = 16 step
              const uint32_t ta = tmem_base + (uint32_t)(P_TMEM_COL + kc * (KC / 2));
#pragma unroll
              for (int k = 0; k < KC / 16; ++k) tc_mma_ts(tmem_s, ta + (uint32_t)(8 * k), bd + (uint64_t)(2 * k), idesc, (kc | k) ? 1u : 0u);
              if (!dbg_noTma) tc_commit(&bars.w_empty[stage]);
              if (kc == NKC - 1) tc_commit(&bars.s_full[wg]);
            }
            __syncwarp();
            FFC_PROF_T(q4);
            FFC_PROF_ADD(prof_c, q3, q4);
            if (++stage == NS1) {
              stage = 0;
              ph ^= 1;
            }
          }
        }
        ++ni;
        if (lane == 0) FFC_STAMP(3);
      }
      if (lane == 0) {
        FFC_PROF_STORE(0, prof_a);
        FFC_PROF_STORE(1, prof_b);
        FFC_PROF_STORE(2, prof_c);
      }
    } else if (warp >= 4) {
      // ---- epilogue: warpgroup g takes the CTA's tiles gi with gi % NEPI == g (S buffer gi % NSB, P~ buffer gi % NPB == g) ----
      const int g = (warp - 4) >> 2;
      const int q4 = warp & 3;                    // TMEM lane quarter
      const int r_local = q4 * 32 + lane;         // row within the item
      const float a2 = prm.a2, b2 = prm.b2;
      const int k = prm.k;
      uint32_t* scan_stage = reinterpret_cast<uint32_t*>(sW1 + NS1 * CHUNK1_BYTES) + (warp - 4) * 32;   // 128 bytes per epilogue warp
      // end-of-item staging of warpgroups 1 and 2 (own region: the W ring is being refilled for the next item by then)
      unsigned char* item_stage = sW1 + NS1 * CHUNK1_BYTES + SCAN_STAGE_BYTES;
      float* stage_l = reinterpret_cast<float*>(item_stage);                                           // [2][128]
      float* stage_v = reinterpret_cast<float*>(item_stage + (NEPI - 1) * BM * 4);                     // [2][128][KMAX]
      int32_t* stage_i = reinterpret_cast<int32_t*>(item_stage + (NEPI - 1) * BM * 4 * (1 + KMAX));    // [2][128][KMAX]
      const uint32_t pt_remote0 = map_to_rank(smem_u32(smem + OFF_DATA), 1);
      const uint32_t ptfull_remote0 = map_to_rank(smem_u32(&bars.pt_full[0]), 1);
      uint32_t s_use = 0;       // tiles this warpgroup has taken so far (all items): phase of s_full[g]
      uint32_t gi0 = 0;         // the CTA's tile count at the start of the current item
      uint32_t hi0 = 0;         // ... counting only tiles handed to the O-CTA (not those of hard-negative-only items): tile h uses P~ buffer h % NPB
      FFC_PROF_DECL(prof_e0);
      FFC_PROF_DECL(prof_e1);
      FFC_PROF_DECL(prof_e2);
      FFC_PROF_DECL(prof_trig);
      for (int ia = pair; ia < n_items; ia += n_pairs) {
        const Item it = decode_item(prm, ia);
        const SubSweep& sw = prm.sub[it.sidx];
        const int sidx = it.sidx, chunk = it.chunk, row0 = it.row0, t_begin = it.t_begin, n_tiles = it.n_tiles;
        const int64_t n_cols = it.n_cols;
        // sweep position -> probe row: with a row map the rows are swept in "positives first, hard-negative-only rows last" order
        const int pos = row0 + r_local;
        const bool row_ok = pos < prm.n_rows;
        const int row = row_ok ? (prm.row_map ? prm.row_map[pos] : pos) : 0;
        const bool all_out = it.all_out;
        if (n_tiles == 0) {
          // an item without columns still owes its l / top-k partials (zeros / -inf)
          if (g == 0 && row_ok) {
            const int64_t pr = (int64_t)chunk * prm.n_rows + row;
            sw.l_part[pr] = 0.f;
            for (int q = 0; q < k; ++q) {
              sw.topv_part[pr * k + q] = -INFINITY;
              sw.topi_part[pr * k + q] = -1;
            }
          }
          continue;
        }
        const int32_t tcol = (row_ok && sw.tcol) ? sw.tcol[row] : -1;
        const bool outl = row_ok && prm.is_out && prm.is_out[row];
        const bool warp_out = __any_sync(0xffffffffu, outl);
        float thr = INFINITY;
        if (SV && row_ok && sw.thr) thr = sw.thr[row];
        float lsum = 0.f;
        // hard-negative top-k state of this row (see topk_scan16)
        int tk[KMAX], tc[KMAX];
#pragma unroll
        for (int q = 0; q < KMAX; ++q) {
          tk[q] = 0;
          tc[q] = -1;
        }
        int kth = 0;
        // Threshold shared by the work items of the same probe rows (one per column chunk): the k-th largest cosine any of them
        // has seen so far is a lower bound of the row's final k-th, so nothing at or below it can enter the merged top-k.  Each
        // item publishes its own k-th (atomicMax on the integer key) and picks the maximum up at every tile: the candidate rate
        // of an item falls as if it had seen all chunks' columns.  Main sweep only (the side sets merge per loss).
        int32_t* kshare = (sidx == 0 && outl) ? prm.kth_shared + row : nullptr;
        int kfloor = 0, kpub = 0;
        float pthr = __uint_as_float(__float_as_uint(ex2f(-b2)) & 0xffff0000u);    // p~ of cosine 0, rounded down to bf16
        if (!dbg_noS) {
          // probe tile -> TMEM (the A operand of every GEMM-1 of this item): thread = row, 32 columns (64 bf16, 128 bytes) per store; the
          // three warpgroups take the 32-column pieces round-robin.  Every GEMM-1 of the previous item has completed: its epilogue
          // warps met at the end-of-item barrier after their last s_full.
          const uint4* src = reinterpret_cast<const uint4*>(prm.p16 + (int64_t)(row_ok ? row : 0) * D);
          const uint32_t tp = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)P_TMEM_COL;
#pragma unroll 1
          for (int c0 = 32 * g; c0 < D / 2; c0 += 32 * NEPI) {
            uint32_t v[32];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const uint4 t = row_ok ? __ldg(src + c0 / 4 + q) : make_uint4(0u, 0u, 0u, 0u);
              v[4 * q] = t.x;
              v[4 * q + 1] = t.y;
              v[4 * q + 2] = t.z;
              v[4 * q + 3] = t.w;
            }
            tc_st32(tp + (uint32_t)c0, v);
          }
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bars.p_full);
        }
        if (sidx == 0 && warp_out && prm.done_flags) {
          // Seed the row's list with the hard negatives that FINISHED items of the same probe rows (other column chunks, earlier waves
          // of the grid) have already found: entries with column -2, dropped again when the item's own partial is written.  The
          // list's k-th is then the exact k-th over all finished columns plus this item's, instead of starting from zero -- without
          // it an item only learns from its own columns, and at the 8-way shard shape 70 % of the 32-column chunks of an outlier-heavy
          // batch ran the exact scan (27 % with the seeds; profiles/r2_outlier_sweep.md).  Runs while the first GEMM-1 is in flight.
          const int n_row_tiles = (prm.n_rows + BM - 1) / BM;
          const int32_t* flag = prm.done_flags + row0 / BM;
          for (int c2 = 0; c2 < sw.n_chunks; ++c2) {
            if (c2 == chunk) continue;
            int f;
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(f) : "l"(flag + (int64_t)c2 * n_row_tiles) : "memory");
            if (f != prm.epoch || !outl) continue;
            const float* pv = sw.topv_part + ((int64_t)c2 * prm.n_rows + row) * k;
            float xs[KMAX];
#pragma unroll
            for (int q = 0; q < KMAX; ++q) xs[q] = q < k ? __ldcg(pv + q) : -INFINITY;      // independent loads, one round trip
#pragma unroll
            for (int q = 0; q < KMAX; ++q) {
              const int xk = (int)(__float_as_uint(xs[q]) & TOPK_VAL_MASK);
              if (xs[q] > 0.f && xk > kth) {      // (sorted: once one fails the rest does too)
                topk_insert_key(xk, -2, k, tk, tc);
#pragma unroll
                for (int r = 0; r < KMAX; ++r)
                  if (r == k - 1) kth = tk[r];
              }
            }
          }
          if (outl) {
            if (kth > 0) {
              atomicMax(kshare, kth);
              kpub = kth;
            }
          }
        }
        const int first = (g + NEPI - (int)(gi0 % NEPI)) % NEPI;      // this warpgroup's first tile of the item
        for (int i = first; i < n_tiles; i += NEPI, ++s_use) {
          const int sb = (int)((gi0 + (uint32_t)i) & (NSB - 1));
          const int j0 = (t_begin + i) * BN;
          // exclusion words of the four 32-column chunks of this tile (one 16-byte load, issued before the waits)
          uint4 cm = make_uint4(0u, 0u, 0u, 0u);
          if (sw.cmask && (int64_t)j0 < n_cols) cm = __ldg(reinterpret_cast<const uint4*>(sw.cmask + (j0 >> 5)));
          int kshared = 0;
          if (kshare) kshared = __ldcg(kshare);
          FFC_PROF_T(e0);
          // s_full is per warpgroup: this is the warpgroup's s_use-th tile.  (Per-buffer barriers would be waited by
          // different warpgroups in turn; with fewer S buffers than warpgroups + 1 a slow warpgroup gets lapped by a phase and
          // a parity wait two phases behind never returns.)
          mbar_wait(&bars.s_full[g], s_use & 1);
          tc_fence_after();
          FFC_PROF_T(e1);
          const uint32_t hi = hi0 + (uint32_t)i;          // the tile's number among the tiles handed to the O-CTA
          const int pb = (int)(hi % NPB);
          const bool hand = !dbg_noHand && !all_out;
          if (hand) mbar_wait_cluster(&bars.pt_empty[pb], ((hi / NPB) & 1) ^ 1);
          FFC_PROF_T(e2);
          FFC_PROF_ADD(prof_e0, e0, e1);
          FFC_PROF_ADD(prof_e1, e1, e2);
          const uint32_t tmem_s = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(sb * BN);
          const uint32_t pt_remote = pt_remote0 + (uint32_t)(pb * PT_BYTES);
          const uint32_t ptfull_remote = ptfull_remote0 + (uint32_t)(pb * 8);
          // One loop over the tile's four 32-column chunks.  Exclusions (a `ones` column, the row's target, the ragged tail) are
          // decided per CHUNK and warp-uniformly: only chunks that hold one pay for the per-element test, the others are pure
          // ld -> ex2 -> pack -> st.async.  (At 8-way shard shapes ~60 % of the TILES hold a `ones` column, but only ~20 % of
          // the chunks.)
          kfloor = max(kfloor, kshared);
          kth = max(kth, kfloor);
          if (!SV && !all_out && warp_out) pthr = __uint_as_float(__float_as_uint(ex2f(fmaf(__int_as_float(kth & (int)TOPK_VAL_MASK), a2, -b2))) & 0xffff0000u);
          float l0 = 0.f, l1 = 0.f;
#pragma unroll 1
          for (int cc = 0; cc < BN / 32; ++cc) {
            uint32_t v[32];
            if (dbg_noEpi) {
#pragma unroll
              for (int c = 0; c < 32; ++c) v[c] = 0u;
            } else {
              tc_ld32(tmem_s + cc * 32, v);
            }
            if (cc == BN / 32 - 1) {      // S buffer sb is in registers now: a later tile's MMA may overwrite it
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(&bars.s_empty[sb]);
            }
            const int col0 = j0 + cc * 32;
            uint32_t excl = cc == 0 ? cm.x : cc == 1 ? cm.y : cc == 2 ? cm.z : cm.w;
            const int trel = tcol - col0;
            if ((unsigned)trel < 32u) excl |= 1u << trel;
            if ((int64_t)col0 + 32 > n_cols) {
              const int nv = (int)(n_cols - col0);   // valid columns in this chunk (may be <= 0)
              excl |= nv <= 0 ? 0xffffffffu : (0xffffffffu << nv);
            }
            const bool slow = __any_sync(0xffffffffu, excl != 0u);
            uint32_t pk[16];
            // (hard-negative-only items: no softmax term -- ffc.py:86-92 takes the top-k of the raw cosines and nothing else from these
            // rows -- so no exponentials, no P~ tile, and the O-CTA sits the item out)
            if constexpr (DQ_SV) {
              // column col0 + lane's (thr_1, thr_2, a_1, a_2), handed to the 32 rows of the warp column by column (a = 0 past the
              // last column and on hard-negative-only rows).  The two losses' p~ differ only where their hardness does, so one
              // exponential per element unless the column's thresholds differ (warp-uniform).
              const float4 cw = (int64_t)col0 + lane < n_cols ? __ldg(prm.dq_col + col0 + lane) : make_float4(INFINITY, INFINITY, 0.f, 0.f);
  #pragma unroll
              for (int c = 0; c < 32; c += 2) {
                float w[2];
  #pragma unroll
                for (int e = 0; e < 2; ++e) {
                  const float t1 = __shfl_sync(0xffffffffu, cw.x, c + e), t2 = __shfl_sync(0xffffffffu, cw.y, c + e);
                  const float c1 = __shfl_sync(0xffffffffu, cw.z, c + e), c2 = __shfl_sync(0xffffffffu, cw.w, c + e);
                  const float x = __uint_as_float(v[c + e]);
                  const bool m1 = x > t1;
                  const float p1 = ex2f(fmaf(m1 ? fmaf(SV_T, x, SV_T - 1.f) : x, a2, -b2)) * (m1 ? SV_T : 1.f);
                  if (t1 == t2) {
                    w[e] = (c1 + c2) * p1;
                  } else {
                    const bool m2 = x > t2;
                    const float p2 = ex2f(fmaf(m2 ? fmaf(SV_T, x, SV_T - 1.f) : x, a2, -b2)) * (m2 ? SV_T : 1.f);
                    w[e] = fmaf(c1, p1, c2 * p2);
                  }
                }
                l0 += w[0];
                l1 += w[1];
                pk[c >> 1] = pack_bf16(w[0], w[1]);
              }
            } else if (!all_out) {
  #pragma unroll
              for (int c = 0; c < 32; c += 2) {
                if (dbg_noEpi) {
                  pk[c >> 1] = 0u;
                  continue;
                }
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
                if (slow) {   // warp-uniform: only chunks that contain an excluded column pay for the per-element test
                  if ((excl >> c) & 1u) p0 = g0 = 0.f;
                  if ((excl >> (c + 1)) & 1u) p1 = g1 = 0.f;
                }
                l0 += p0;
                l1 += p1;
                pk[c >> 1] = pack_bf16(g0, g1);
              }
            }
            // ---- hard-negative top-k on the raw cosines of outlier rows ----
            if (SV) {
              if (warp_out) {
                topk_scan16<0, 32>(v, excl & 0xffffu, col0, outl, k, tk, tc, kth, kfloor);
                topk_scan16<16, 32>(v, excl >> 16, col0 + 16, outl, k, tk, tc, kth, kfloor);
              }
            } else if (warp_out) {
              // Without SV, p~ is monotonic in the cosine: the chunk can only hold a candidate if the maximum of its packed p~ (one
              // bf16x2 max tree; excluded columns are 0) reaches the row's threshold mapped to p~ space.
              bool mine;
              if (all_out) {      // no p~ here: the raw cosines' bit patterns (an excluded column can only cause a needless exact scan)
                int mx = (int)v[0];
#pragma unroll
                for (int c = 1; c < 32; ++c) mx = max(mx, (int)v[c]);
                mine = outl && (mx | 31) > kth;      // (| 31: a key carries the column index in the low bits)
              } else {
                uint32_t m = pk[0];
#pragma unroll
                for (int q = 1; q < 16; ++q) m = max_bf16x2(m, pk[q]);
                const float mf = fmaxf(__uint_as_float(m << 16), __uint_as_float(m & 0xffff0000u));
                mine = outl && mf >= pthr;
              }
              unsigned cand = __ballot_sync(0xffffffffu, mine);
              if (cand) {
                FFC_PROF_ADD(prof_trig, 0, 1);
                if (__popc(cand) > 4) {      // many rows at once (the first tiles of an item): the per-lane scan is cheaper
                  topk_scan16<0, 32>(v, excl & 0xffffu, col0, outl, k, tk, tc, kth, kfloor);
                  topk_scan16<16, 32>(v, excl >> 16, col0 + 16, outl, k, tk, tc, kth, kfloor);
                  cand = 0u;
                }
                // Usually ONE lane (row) has a candidate: its 32 cosines go through shared memory so that the 32 lanes test one
                // column each; the row's lane then inserts the (usually single) hit.  ~40 instructions instead of a 32-key scan.
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
                // threshold in p~ space, rounded DOWN to bf16 (the packed values are rounded to nearest): never misses a candidate
                if (!all_out) pthr = __uint_as_float(__float_as_uint(ex2f(fmaf(__int_as_float(kth & (int)TOPK_VAL_MASK), a2, -b2))) & 0xffff0000u);
              }
            }
            // P~[r_local][cc*32 .. +32) = 4 pieces of 16 bytes; each st.async counts itself on the peer's pt_full[pb]
            if (hand) {
#pragma unroll
              for (int q = 0; q < 4; ++q)
                st_async_v4(pt_remote + pt_offset((uint32_t)(cc * 4 + q), (uint32_t)r_local), ptfull_remote, pk[4 * q], pk[4 * q + 1], pk[4 * q + 2],
                            pk[4 * q + 3]);
            }
          }
          lsum += l0 + l1;
          if (kshare) {      // publish this item's own k-th when it has risen
            int kown = 0;
#pragma unroll
            for (int r = 0; r < KMAX; ++r)
              if (r == k - 1) kown = tk[r];
            if (kown > kpub) {
              atomicMax(kshare, kown);
              kpub = kown;
            }
          }
          FFC_PROF_T(e3);
          FFC_PROF_ADD(prof_e2, e2, e3);
        }
        gi0 += (uint32_t)n_tiles;
        if (!all_out) hi0 += (uint32_t)n_tiles;
        // ---- per-row partials: combine the three warpgroups through shared memory ----
        // Named barrier 1 (the 12 epilogue warps): every warpgroup has seen its last s_full of the item, i.e. every GEMM-1 that reads
        // this item's P has completed (the next item's P may be stored), and the previous item's staging has been consumed.
        asm volatile("bar.sync 1, 384;" ::: "memory");
        float tv[KMAX];
        int32_t ti[KMAX];
#pragma unroll
        for (int q = 0; q < KMAX; ++q) {
          const bool live = tk[q] > 0 && tc[q] >= 0;      // (column -2: a seed from another item's partial -- it is reported there)
          tv[q] = live ? __int_as_float(tk[q] & (int)TOPK_VAL_MASK) : -INFINITY;
          ti[q] = live ? tc[q] + (tk[q] & 31) : -1;
        }
        if (g >= 1) {
          stage_l[(g - 1) * BM + r_local] = lsum;
#pragma unroll
          for (int q = 0; q < KMAX; ++q) {
            stage_v[((g - 1) * BM + r_local) * KMAX + q] = tv[q];
            stage_i[((g - 1) * BM + r_local) * KMAX + q] = ti[q];
          }
        }
        asm volatile("bar.sync 1, 384;" ::: "memory");
        if (g == 0 && row_ok) {
#pragma unroll 1
          for (int og = 0; og < NEPI - 1; ++og) lsum += stage_l[og * BM + r_local];
          if (outl) {
            // the own list may have holes where seeds were: rebuild it by insertion, then merge the other warpgroups' lists
            float ov[KMAX];
            int32_t oi[KMAX];
#pragma unroll
            for (int q = 0; q < KMAX; ++q) {
              ov[q] = tv[q];
              oi[q] = ti[q];
              tv[q] = -INFINITY;
              ti[q] = -1;
            }
            float kthv = -INFINITY;
#pragma unroll
            for (int q = 0; q < KMAX; ++q) {
              if (q < k && ov[q] > kthv) {
                topk_insert<KMAX>(tv, ti, k, ov[q], oi[q]);
#pragma unroll
                for (int qq = 0; qq < KMAX; ++qq)
                  if (qq == k - 1) kthv = tv[qq];
              }
            }
#pragma unroll 1
            for (int og = 0; og < NEPI - 1; ++og) {
#pragma unroll 1
              for (int q = 0; q < k; ++q) {
                const float x = stage_v[(og * BM + r_local) * KMAX + q];
                if (x > kthv) {
                  topk_insert<KMAX>(tv, ti, k, x, stage_i[(og * BM + r_local) * KMAX + q]);
#pragma unroll
                  for (int qq = 0; qq < KMAX; ++qq)
                    if (qq == k - 1) kthv = tv[qq];
                }
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
          __threadfence();      // the partial is visible before the item is flagged finished (below)
        }
        if (sidx == 0 && prm.done_flags && g == 0) {
          asm volatile("bar.sync 4, 128;" ::: "memory");      // warpgroup 0: all 128 rows' partials are out
          if (warp == 4 && lane == 0) {
          const int n_row_tiles = (prm.n_rows + BM - 1) / BM;
            asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(prm.done_flags + (int64_t)chunk * n_row_tiles + row0 / BM), "r"(prm.epoch) : "memory");
          }
        }
      }
      if (warp == 4 && lane == 0) {
        FFC_PROF_STORE(3, prof_e0);
        FFC_PROF_STORE(4, prof_e1);
        FFC_PROF_STORE(5, prof_e2);
        FFC_PROF_STORE(7, prof_trig);
      }
    }
  } else {
    // =========================================== O-CTA ===========================================
    if (warp == 0) {
      // ---- TMA producer: one 3-D box (64 features x JB queue rows x D/64 feature chunks) per stage ----
      int stage = 0;
      uint32_t ph = 0;
      FFC_PROF_DECL(prof_tma);
      for (int ia = pair; ia < n_items; ia += n_pairs) {
        const Item it = decode_item(prm, ia);
        if (it.n_tiles == 0 || it.all_out || dbg_noO || dbg_noTma) continue;
        const CUtensorMap* map_w2 = it.sidx == 0 ? &map_w2a : (it.sidx == 1 ? &map_w2b : &map_w2c);
        for (int t = it.t_begin; t < it.t_begin + it.n_tiles; ++t) {
#pragma unroll
          for (int jb = 0; jb < BN / JB; ++jb) {
            FFC_PROF_T(q0);
            mbar_wait(&bars.w2_empty[stage], ph ^ 1);
            FFC_PROF_T(q1);
            FFC_PROF_ADD(prof_tma, q0, q1);
            if (elect_one()) {
              mbar_expect_tx(&bars.w2_full[stage], (uint32_t)Sh::STAGE2_BYTES);
              tma_load_3d(map_w2, &bars.w2_full[stage], sW2 + stage * Sh::STAGE2_BYTES, 0, t * BN + jb * JB, 0);
            }
            __syncwarp();
            if (++stage == Sh::NS2) {
              stage = 0;
              ph ^= 1;
            }
          }
        }
      }
      if (lane == 0) FFC_PROF_STORE(6, prof_tma);
    } else if (warp == 1) {
      // ---- GEMM-2 issue: O[128 x D] += P~[128 x 128] . W_tile[128 x D]; per K = 16 queue rows one MMA per 256 features ----
      constexpr uint32_t idesc = make_idesc(BM, Sh::N2, 0, 1);
      // A = P~: interleaved core matrices, K halves 2 KB apart (LBO), 8-row groups 128 B apart (SBO)
      const uint64_t a0 = make_desc(smem_u32(sPt), BM * 16, 128, 0);
      // B = W stage, MN-major (N = feature dim): 64-feature atoms JB*128 bytes apart (LBO), 8-row groups 1 KB apart (SBO)
      const uint64_t b0 = make_desc(smem_u32(sW2), JB * 128, 1024);
      int stage = 0, pb = 0;
      uint32_t ph = 0, pt_ph = 0;
      uint32_t ni = 0;      // items with tiles so far
      FFC_PROF_DECL(prof_a);
      FFC_PROF_DECL(prof_b);
      FFC_PROF_DECL(prof_c);
      FFC_PROF_DECL(prof_gap);
      for (int ia = pair; ia < n_items; ia += n_pairs) {
        const Item it = decode_item(prm, ia);
        const int n_tiles = it.n_tiles;
        if (n_tiles == 0 || it.all_out) continue;      // (hard-negative-only items have no GEMM-2: the O-CTA sits them out)
        if (ni > 0) {     // the previous item's O has been read out of TMEM by the write-out warps
          FFC_PROF_T(g0);
          mbar_wait(&bars.o_empty, (ni - 1) & 1);
          FFC_PROF_T(g1);
          FFC_PROF_ADD(prof_gap, g0, g1);
        }
        tc_fence_after();
        if (ni == 0 && lane == 0) FFC_STAMP(2);
        for (int i = 0; i < n_tiles; ++i) {
          FFC_PROF_T(q0);
          if (!dbg_noHand) mbar_wait(&bars.pt_ready[pb], pt_ph);     // P~ complete and fenced by the hand-off warp
          tc_fence_after();
          FFC_PROF_T(q1);
          FFC_PROF_ADD(prof_a, q0, q1);
          // the P~ buffer of the item's LAST tile is not released here: the write-out warps stage O through it and release it
          const bool release_pt = i + 1 < n_tiles && !dbg_noHand;
          if (dbg_noO) {
            if (release_pt && elect_one()) mbar_arrive_remote(map_to_rank(smem_u32(&bars.pt_empty[pb]), 0));
            __syncwarp();
          } else {
            const uint64_t ap = a0 + (uint64_t)(pb * (PT_BYTES >> 4));
#pragma unroll
            for (int jb = 0; jb < BN / JB; ++jb) {
              FFC_PROF_T(q2);
              if (!dbg_noTma) {
                mbar_wait(&bars.w2_full[stage], ph);
                tc_fence_after();
              }
              FFC_PROF_T(q3);
              FFC_PROF_ADD(prof_b, q2, q3);
              if (elect_one()) {
                const uint64_t bs = b0 + (uint64_t)(stage * (Sh::STAGE2_BYTES >> 4));
#pragma unroll
                for (int k16 = 0; k16 < JB / 16; ++k16) {
                  const int kk = jb * JB + k16 * 16;                                    // queue row within the tile
                  const uint64_t ad = ap + (uint64_t)((kk >> 3) * ((BM * 16) >> 4));
#pragma unroll
                  for (int nh = 0; nh < Sh::NHALF; ++nh) {
                    const uint64_t bd = bs + (uint64_t)(nh * 4 * ((JB * 128) >> 4) + k16 * ((16 * 128) >> 4));
                    tc_mma(tmem_base + (uint32_t)(nh * 256), ad, bd, idesc, (i | jb | k16) ? 1u : 0u);
                  }
                }
                if (!dbg_noTma) tc_commit(&bars.w2_empty[stage]);
                // frees P~ buffer pb: arrives in the S-CTA (cluster rank 0)
                if (jb == BN / JB - 1 && release_pt) tc_commit_mcast(&bars.pt_empty[pb], (uint16_t)1);
              }
              __syncwarp();
              FFC_PROF_T(q4);
              FFC_PROF_ADD(prof_c, q3, q4);
              if (++stage == Sh::NS2) {
                stage = 0;
                ph ^= 1;
              }
            }
          }
          if (++pb == NPB) {
            pb = 0;
            pt_ph ^= 1;
          }
        }
        if (elect_one()) {
          if (dbg_noO) mbar_arrive(&bars.o_full); else tc_commit(&bars.o_full);
        }
        __syncwarp();
        if (lane == 0) FFC_STAMP(3);
        mbar_wait(&bars.o_full, ni & 1);     // one polling warp; the 8 write-out warps block on a hardware barrier instead
        __syncwarp();
        asm volatile("bar.sync 2, 288;" ::: "memory");
        ++ni;
      }
      if (lane == 0) {
        FFC_PROF_STORE(0, prof_a);
        FFC_PROF_STORE(1, prof_b);
        FFC_PROF_STORE(2, prof_c);
        FFC_PROF_STORE(7, prof_gap);
      }
    } else if (warp == 3) {
      // ---- P~ hand-off: wait for the peer's 32 KB (st.async complete_tx bytes), make the generic-proxy writes visible to the
      // async proxy (tcgen05.mma reads P~ through it) and pass the buffer on.  The fence costs 200-1100 cycles while TMA
      // loads are in flight, so it lives here and not in the MMA warp.
      int pb = 0;
      uint32_t pt_ph = 0;
      for (int ia = pair; ia < n_items; ia += n_pairs) {
        const Item it = decode_item(prm, ia);
        if (dbg_noHand) break;
        if (it.all_out) continue;
        for (int i = 0; i < it.n_tiles; ++i) {
          if (elect_one()) mbar_expect_tx(&bars.pt_full[pb], PT_BYTES);     // the single arriver of pt_full[pb]
          __syncwarp();
          mbar_wait_cluster(&bars.pt_full[pb], pt_ph);
          asm volatile("fence.proxy.async;" ::: "memory");
          __syncwarp();
          if (elect_one()) mbar_arrive(&bars.pt_ready[pb]);
          __syncwarp();
          if (++pb == NPB) {
            pb = 0;
            pt_ph ^= 1;
          }
        }
      }
    } else if (warp >= 4 && warp < 12) {
      // ---- O write-out: TMEM -> global partial [chunk][row][D]; warpgroup g takes half of the columns ----
      const int g = (warp - 4) >> 2;
      const int q4 = warp & 3;
      constexpr int half = D / 2;                  // D is a multiple of 64
      uint32_t gtiles = 0;      // the CTA's tile count at the start of the current item
      for (int ia = pair; ia < n_items; ia += n_pairs) {
        const Item it = decode_item(prm, ia);
        const SubSweep& sw = prm.sub[it.sidx];
        const int row0 = it.row0, n_tiles = it.n_tiles;
        if (it.all_out) continue;      // no O partial: the finalize kernels never read the O sums of a hard-negative-only row
        // destination rows: lane l keeps the probe row of sweep position row0 + q4*32 + l (or -1), handed round by shuffle
        const int my_pos = row0 + q4 * 32 + lane;
        const int my_row = my_pos < prm.n_rows ? (prm.row_map ? prm.row_map[my_pos] : my_pos) : -1;
        float* dst_col = sw.o_part + (int64_t)it.chunk * prm.n_rows * D + g * half;
        if (n_tiles == 0) {
          // an item without columns owes a zero partial (4 rows x 128 B per store instruction)
          for (int c0 = 0; c0 < half; c0 += 32) {
#pragma unroll
            for (int itr = 0; itr < 8; ++itr) {
              const int r = itr * 4 + (lane >> 3), c = (lane & 7) * 4;
              const int orow = __shfl_sync(0xffffffffu, my_row, r);
              if (orow >= 0) *reinterpret_cast<uint4*>(dst_col + (int64_t)orow * D + c0 + c) = make_uint4(0u, 0u, 0u, 0u);
            }
          }
          continue;
        }
        asm volatile("bar.sync 2, 288;" ::: "memory");   // released by the MMA warp once every tcgen05.mma of the item has completed
        tc_fence_after();
        // A TMEM lane is a row, so a thread holds 32 consecutive floats of ITS row: stored straight from the registers every store
        // instruction touched 32 different 2 KB-strided rows, 16 bytes each (the write-out took 12-17 us per item).  Each warp
        // transposes its 32 x 32 block through 4 KB of shared memory instead -- 16-byte pieces XOR-swizzled by the row, so both the
        // row-wise writes and the reads are conflict-free -- and a store instruction then covers 4 rows x 128 contiguous bytes.
        // The 8 x 4 KB are the P~ buffer of the item's last tile: its MMAs have completed, and the S-CTA may not refill it until the
        // write-out warps release it below (its two other buffers are already being filled for the next item).
        const int pb_last = (int)((gtiles + (uint32_t)n_tiles - 1u) % NPB);
        unsigned char* stg = sPt + pb_last * PT_BYTES + (warp - 4) * 4096;
        for (int c0 = 0; c0 < half; c0 += 32) {
          uint32_t v[32];
          tc_ld32(tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(g * half + c0), v);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<uint4*>(stg + lane * 128 + ((q ^ (lane & 7)) << 4)) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          __syncwarp();
#pragma unroll
          for (int itr = 0; itr < 8; ++itr) {
            const int r = itr * 4 + (lane >> 3), c = lane & 7;
            const uint4 x = *reinterpret_cast<const uint4*>(stg + r * 128 + ((c ^ (r & 7)) << 4));
            const int orow = __shfl_sync(0xffffffffu, my_row, r);
            if (orow >= 0) *reinterpret_cast<uint4*>(dst_col + (int64_t)orow * D + c0 + c * 4) = x;
          }
          __syncwarp();
        }
        tc_fence_before();
        asm volatile("bar.sync 3, 256;" ::: "memory");      // the 8 write-out warps: O is out of TMEM, the staging buffer is idle
        if (warp == 4) {
          if (elect_one()) {
            mbar_arrive(&bars.o_empty);
            if (!dbg_noHand) mbar_arrive_remote(map_to_rank(smem_u32(&bars.pt_empty[pb_last]), 0));
          }
          __syncwarp();
        }
        gtiles += (uint32_t)n_tiles;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) FFC_STAMP(4);
  cluster_sync_all();     // the peer may still signal into this CTA's shared memory until here
  if (warp == 2) {
    const uint32_t ncols = rank == 0 ? 512u : (uint32_t)(D < 32 ? 32 : D);
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ncols) : "memory");
  }
  if (threadIdx.x == 0) {
    FFC_STAMP(5);
    FFC_STAMP_NS(7);
  }
}

// ------------------------------------------------------------------------------------------------
// host side: tensor maps + launch
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct MapKey {
  const void* ptr;
  int64_t rows;
  int D, box_rows;
  bool operator==(const MapKey& o) const { return ptr == o.ptr && rows == o.rows && D == o.D && box_rows == o.box_rows; }
};
struct Sm100Cache {
  PFN_encodeTiled encode = nullptr;
  std::vector<std::pair<MapKey, CUtensorMap>> maps;
  int32_t* done_flags = nullptr;     // [column chunk][row tile] item-finished flags of the main sweep (value = the launch's epoch)
  int64_t done_cap = 0;
  int epoch = 0;
};

Sm100Cache* sm100_cache_create() { return new Sm100Cache(); }
void sm100_cache_destroy(Sm100Cache* c) {
  if (c && c->done_flags) cudaFree(c->done_flags);
  delete c;
}

int sm100_get_map(Sm100Cache* c, const void* ptr, int64_t rows, int D, int box_rows, bool chunked3d, CUtensorMap* out) {
  MapKey key{ptr, rows, D, chunked3d ? -box_rows : box_rows};
  for (auto& e : c->maps)
    if (e.first == key) {
      *out = e.second;
      return FFC_OK;
    }
  if (!c->encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    FFC_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    FFC_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available in this driver");
    c->encode = (PFN_encodeTiled)fn;
  }
  CUtensorMap m;
  CUresult r;
  if (!chunked3d) {
    // [rows, D] bf16 row-major; box = 64 features (one 128-byte swizzle row) x box_rows
    cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)D * 2};
    cuuint32_t box[2] = {(cuuint32_t)KC, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    r = c->encode(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  } else {
    // the same matrix seen as [D/64 chunks][rows][64]: one box = (64 features, box_rows rows, all D/64 chunks) lands in
    // shared memory chunk-major, i.e. D/64 consecutive [box_rows x 128 B] swizzled slabs -- a whole GEMM-2 stage per TMA
    cuuint64_t dims[3] = {(cuuint64_t)KC, (cuuint64_t)rows, (cuuint64_t)(D / KC)};
    cuuint64_t strides[2] = {(cuuint64_t)D * 2, (cuuint64_t)KC * 2};
    cuuint32_t box[3] = {(cuuint32_t)KC, (cuuint32_t)box_rows, (cuuint32_t)(D / KC)};
    cuuint32_t estr[3] = {1, 1, 1};
    r = c->encode(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with %d (ptr=%p rows=%lld D=%d box_rows=%d 3d=%d)", (int)r, ptr, (long long)rows, D, box_rows, (int)chunked3d);
    return FFC_ERR_CUDA;
  }
  if (c->maps.size() > 64) c->maps.clear();
  c->maps.emplace_back(key, m);
  *out = m;
  return FFC_OK;
}

// D <= 256 runs on the one-CTA kernel (head_sm100_1cta.cu) unless FFC_SWEEP_PAIR=1 asks for the CTA-pair kernel (A/B measurements)
static bool use_one_cta(int D) {
  static const bool force_pair = getenv("FFC_SWEEP_PAIR") != nullptr && atoi(getenv("FFC_SWEEP_PAIR")) != 0;
  return D <= 256 && !force_pair;
}

// CTA pairs that can be resident at once (one CTA per SM, both CTAs of a pair on one TPC): the persistent grid
static int pair_slots() {
  static int slots = 0;
  if (!slots) {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms >= 2) slots = sms / 2;
    else slots = 74;
    const char* e = getenv("FFC_SWEEP_PAIRS");
    if (e && atoi(e) > 0) slots = atoi(e);
  }
  return slots;
}
// Launch shape of the CTA-pair kernel.  Default: one pair per item, dealt to the SMs by the hardware (the kernel's item loop runs once).
// FFC_SWEEP_PERSISTENT=1 (or a pair count forced with FFC_SWEEP_PAIRS): with more than 2 x slots items the grid is `slots` persistent
// pairs that walk the item list, so that set-up, P load and O write-out of consecutive items overlap.  Measured at the 2 / 4 / 8-way
// shard shapes (profiles/r2_persistent_sweep.md) it is no faster: the steady state is bound by L2 -> SM delivery of W (13.4 TB/s,
// both CTAs of every pair stream every tile), the turn-around it removes was overlapped with other pairs' tiles anyway, and the
// hardware's dynamic dealing balances the short side items better than a static round-robin.  Kept as a tested option.
static bool persistent_grid(int n_items) {
  static const bool on = (getenv("FFC_SWEEP_PERSISTENT") != nullptr && atoi(getenv("FFC_SWEEP_PERSISTENT")) != 0) ||
                         (getenv("FFC_SWEEP_PAIRS") != nullptr && atoi(getenv("FFC_SWEEP_PAIRS")) > 0);
  return on && n_items > 2 * pair_slots();
}
// Pairs of the persistent grid.  FFC_SWEEP_RESERVE (pairs, default 0) leaves TPCs to the kernels that run underneath a sweep on other
// streams (LRU / label bookkeeping, the label prefetch's collectives): a grid that never gives an SM back pushes them behind the whole sweep.
static int persistent_pairs() {
  static const int reserve = getenv("FFC_SWEEP_RESERVE") ? atoi(getenv("FFC_SWEEP_RESERVE")) : 0;
  const int slots = pair_slots();
  return slots > 8 ? std::max(8, slots - std::max(0, reserve)) : slots;
}

int sm100_pick_chunks(int n_rows, int64_t n_cols, int D, int chunk_cap) {
  // items = row_tiles x chunks run as CTA pairs, 74 pairs at a time (one-CTA kernel: 148 CTAs): pick the chunk count whose last
  // wave is fullest (ties -> fewer chunks: fewer partials and fewer P loads / O write-outs)
  const bool one = use_one_cta(D);
  const int slots = one ? 148 : pair_slots();
  static const int forced = getenv("FFC_SWEEP_CHUNKS") ? atoi(getenv("FFC_SWEEP_CHUNKS")) : 0;     // tests: a fixed chunk count
  if (forced > 0) return (int)std::min<int64_t>(std::min(forced, std::max(1, chunk_cap)), std::max<int64_t>(1, ceil_div64(n_cols, one ? sm100_1cta_tile_cols(D) : BN)));
  const int tile_cols = one ? sm100_1cta_tile_cols(D) : BN;
  const int row_tiles = std::max(1, (n_rows + BM - 1) / BM);
  const int64_t n_tiles = std::max<int64_t>(1, ceil_div64(n_cols, tile_cols));
  const int max_c = (int)std::min<int64_t>(n_tiles, std::max(1, std::min(chunk_cap, 40)));      // chunk_cap: what the caller's partial workspace holds
  int best = 1;
  double best_eff = 0.0;
  for (int c = 1; c <= max_c; ++c) {
    const int items = row_tiles * c;
    const bool pers = !one && persistent_grid(items);
    const int slots_c = pers ? persistent_pairs() : slots;
    const int waves = (items + slots_c - 1) / slots_c;
    // every item pays a fixed cost (P load, O write-out and the partial's trip through HBM; one pair per item: also set-up and the
    // cluster launch) worth about 12 tile-times (of 128 columns), about 7 on the persistent grid where consecutive items overlap
    const double fixed = pers ? 7.0 : 12.0;
    const double tiles_per_item = (double)n_tiles / c * tile_cols / 128.0;
    const double eff = ((double)items / (waves * (double)slots_c)) * (tiles_per_item / (tiles_per_item + fixed));
    if (eff > best_eff * 1.005) {
      best_eff = eff;
      best = c;
    }
  }
  return best;
}

template <bool SV, int D, bool DQ_SV = false>
static int launch_one(const CUtensorMap* maps, const Sm100Params& p, int n_items, cudaStream_t s) {
  static bool attr_set = false;
  auto kern = ffc_head_sweep_sm100_kernel<SV, D, DQ_SV>;
  constexpr size_t smem = SweepShape<D>::SMEM;
  if (!attr_set) {
    FFC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  const int n_pairs = persistent_grid(n_items) ? persistent_pairs() : n_items;
  kern<<<dim3(2 * n_pairs), dim3(NTHREADS), smem, s>>>(maps[0], maps[1], maps[2], maps[3], maps[4], maps[5], maps[6], p);
  FFC_LAUNCH_CHECK();
#if FFC_SM100_DEBUG_BUILD
  static int dumps_left = getenv("FFC_SM100_DUMP") ? atoi(getenv("FFC_SM100_DUMP")) : 0;
  if (dumps_left > 0 && n_items >= 64) {
    --dumps_left;
    cudaStreamSynchronize(s);
    FILE* fo = fopen(getenv("FFC_SM100_DUMP_FILE") ? getenv("FFC_SM100_DUMP_FILE") : "gpurun_out/sweep_stamps.log", "a");
    if (!fo) fo = stderr;
    static long long h[1024][8];
    cudaMemcpyFromSymbol(h, g_sweep_stamps, sizeof(h));
    const bool pers = n_pairs < n_items;
    const int main_items = std::min(n_items, p.sub[1].item0);
    const int n = std::min(2 * (pers ? n_pairs : main_items), 1024);     // one pair per item: main-sweep CTAs only
    long long t0 = h[0][6], t1 = 0;
    for (int i = 0; i < n; ++i) {
      t0 = std::min(t0, h[i][6]);
      t1 = std::max(t1, h[i][7]);
    }
    fprintf(fo, "[sweep stamps] debug=%d %d items on %d CTAs%s, kernel %.1f us (globaltimer)\n", p.debug, n_items, 2 * n_pairs, pers ? " (persistent pairs)" : "",
            (t1 - t0) * 1e-3);
    // where an item's time goes (cycles, mean over the CTAs of each role): set-up (barriers, TMEM alloc, cluster sync) | until the
    // MMA loop starts (P into TMEM / first W tile) | MMA loop | after the loop to the end of the role's work (O write-out, partial
    // merge) | final cluster sync + dealloc
    for (int role = 0; role < 2; ++role) {
      double ph[5] = {0, 0, 0, 0, 0};
      int cnt = 0;
      for (int i = role; i < n; i += 2, ++cnt) {
        ph[0] += (double)(h[i][1] - h[i][0]);
        ph[1] += (double)(h[i][2] - h[i][1]);
        ph[2] += (double)(h[i][3] - h[i][2]);
        ph[3] += (double)(h[i][4] - h[i][3]);
        ph[4] += (double)(h[i][5] - h[i][4]);
      }
      fprintf(fo, "  %s-CTA item phases (cycles): set-up %.0f | to MMA loop %.0f | MMA loop %.0f | tail work %.0f | final sync %.0f\n", role ? "O" : "S", ph[0] / cnt,
              ph[1] / cnt, ph[2] / cnt, ph[3] / cnt, ph[4] / cnt);
    }
    static long long hp[1024][8];
    cudaMemcpyFromSymbol(hp, g_sweep_prof, sizeof(hp));
    for (int role = 0; role < 2; ++role) {
      double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      int cnt = 0;
      for (int i = role; i < n; i += 2, ++cnt)
        for (int k = 0; k < 8; ++k) acc[k] += (double)hp[i][k];
      // tiles per CTA (persistent pairs: the main sweep's tiles spread over the pairs; the side items' few tiles are not counted)
      const double nt = pers ? (double)p.sub[0].tiles_per_chunk * main_items / n_pairs : (double)p.sub[0].tiles_per_chunk;
      fprintf(fo, "  %s-CTA cycles/tile: MMA warp waits for %s %.0f, waits for W %.0f, issues %.0f | TMA producer waits %.0f", role ? "O" : "S",
              role ? "P~" : "a free S buffer", acc[0] / cnt / nt, acc[1] / cnt / nt, acc[2] / cnt / nt, acc[6] / cnt / nt);
      if (role == 0)
        fprintf(fo, " | epilogue warp (1 of 3 warpgroups; per tile of the CTA): waits for S %.0f, waits for a free P~ buffer %.0f, works %.0f; top-k scans in %.1f%% of its 32-column chunks", acc[3] / cnt / nt,
                acc[4] / cnt / nt, acc[5] / cnt / nt, 100.0 * acc[7] / cnt / (nt / 3.0 * 4.0));
      if (role == 1) fprintf(fo, " | MMA warp idle between items (O read-out) %.0f per CTA", acc[7] / cnt);
      fprintf(fo, "\n");
    }
    if (fo != stderr) fclose(fo);
  }
#endif
  return FFC_OK;
}

// `sweeps[0 .. n_sweeps)` share P, n_rows, D, is_out, scale, fixed_max, sv and k (taken from sweeps[0]); each has its own
// weight matrix, exclusions, chunk count and partial outputs.
int launch_sweeps_sm100(Sm100Cache* cache, const SweepArgs* sweeps, int n_sweeps, cudaStream_t s) {
  FFC_REQUIRE(n_sweeps >= 1 && n_sweeps <= MAX_SUB, "tcgen05 sweep: %d sweeps per launch (1..%d)", n_sweeps, MAX_SUB);
  if (use_one_cta(sweeps[0].D) && !sweeps[0].force_pair) return launch_sweeps_sm100_1cta(cache, sweeps, n_sweeps, s);
  const SweepArgs& a = sweeps[0];
  FFC_REQUIRE(a.D == 64 || a.D == 128 || a.D == 256 || a.D == 512, "tcgen05 sweep: D=%d must be 64, 128, 256 or 512", a.D);
  FFC_REQUIRE(a.P_bf16, "tcgen05 sweep: bf16 operands missing");
  CUtensorMap maps[1 + 2 * MAX_SUB];
  int rc;
  if ((rc = sm100_get_map(cache, a.P_bf16, a.n_rows, a.D, BM, false, &maps[0]))) return rc;
  Sm100Params p;
  memset(&p, 0, sizeof(p));
  p.n_rows = a.n_rows;
  p.p16 = a.P_bf16;
  p.is_out = a.is_out;
  p.kth_shared = a.kth_shared;
  p.row_map = a.row_map;
  p.n_pos_dev = a.row_map ? a.n_pos_dev : nullptr;
  p.a2 = a.scale * LOG2E;
  p.b2 = a.fixed_max * LOG2E;
  p.k = a.k;
  p.dq_col = a.dq_col;
  p.debug = 0;
#if FFC_SM100_DEBUG_BUILD
  {
    const char* dbg = getenv("FFC_SM100_DEBUG");
    p.debug = dbg ? atoi(dbg) : 0;
  }
#endif
  const int row_tiles = (a.n_rows + BM - 1) / BM;
  int n_items = 0;
  for (int i = 0; i < MAX_SUB; ++i) {
    SubSweep& sb = p.sub[i];
    if (i >= n_sweeps) {       // unused slots: no items, maps duplicated from sweep 0 (never dereferenced)
      sb.item0 = 0x7fffffff;
      maps[1 + 2 * i] = maps[1];
      maps[2 + 2 * i] = maps[2];
      continue;
    }
    const SweepArgs& w = sweeps[i];
    FFC_REQUIRE(w.W_bf16 && w.n_rows == a.n_rows && w.D == a.D && w.P_bf16 == a.P_bf16 && w.sv == a.sv && w.k == a.k && w.n_chunks >= 1,
                "tcgen05 sweep: sweep %d does not share the probe rows / shape of sweep 0", i);
    if ((rc = sm100_get_map(cache, w.W_bf16, w.n_cols, w.D, BN, false, &maps[1 + 2 * i]))) return rc;
    if ((rc = sm100_get_map(cache, w.W2_bf16 ? w.W2_bf16 : w.W_bf16, w.n_cols, w.D, JB, true, &maps[2 + 2 * i]))) return rc;
    sb.n_cols = w.n_cols;
    sb.n_cols_dev = w.n_cols_dev;
    sb.tcol = w.tcol;
    sb.cmask = w.cmask;
    sb.thr = w.thr;
    const int64_t n_tiles = std::max<int64_t>(1, ceil_div64(w.n_cols, BN));
    sb.tiles_per_chunk = (int)ceil_div64(n_tiles, w.n_chunks);
    sb.n_chunks = w.n_chunks;
    sb.item0 = n_items;
    sb.l_part = w.l_part;
    sb.o_part = w.o_part;
    sb.topv_part = w.topv_part;
    sb.topi_part = w.topi_part;
    n_items += row_tiles * w.n_chunks;
  }
  p.n_items = n_items;
  {
    // item-finished flags of the main sweep (seeds of the hard-negative lists): never reset -- a flag counts only if it holds THIS launch's epoch
    const int64_t need = (int64_t)sweeps[0].n_chunks * row_tiles;
    if (need > cache->done_cap) {
      if (cache->done_flags) FFC_CUDA(cudaFree(cache->done_flags));
      cache->done_flags = nullptr;
      cache->done_cap = 0;
      FFC_CUDA(cudaMalloc(&cache->done_flags, (size_t)need * 2 * sizeof(int32_t)));
      FFC_CUDA(cudaMemset(cache->done_flags, 0, (size_t)need * 2 * sizeof(int32_t)));
      cache->done_cap = need * 2;
    }
    static const bool no_seed = getenv("FFC_SWEEP_NO_SEED") != nullptr && atoi(getenv("FFC_SWEEP_NO_SEED")) != 0;      // A/B measurements
    p.done_flags = no_seed ? nullptr : cache->done_flags;
    p.epoch = ++cache->epoch;
    if (cache->epoch == 0x7fffffff) cache->epoch = 0;
  }
#define FFC_SWEEP_CASE(DV)                                                       \
  case DV:                                                                       \
    return a.dq_col ? launch_one<false, DV, true>(maps, p, n_items, s)                    \
                    : (a.sv ? launch_one<true, DV>(maps, p, n_items, s) : launch_one<false, DV>(maps, p, n_items, s));
  switch (a.D) {
    FFC_SWEEP_CASE(64)
    FFC_SWEEP_CASE(128)
    FFC_SWEEP_CASE(256)
    FFC_SWEEP_CASE(512)
  }
#undef FFC_SWEEP_CASE
  return FFC_ERR_INVALID;
}

int launch_sweep_sm100(Sm100Cache* cache, int cache_slot, const SweepArgs& a, cudaStream_t s) {
  (void)cache_slot;
  return launch_sweeps_sm100(cache, &a, 1, s);
}

}  // namespace ffc
