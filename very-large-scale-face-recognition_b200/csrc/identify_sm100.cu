// 1:N identification: the k most similar resident prototypes queue[0][0 .. cur_idx) of every query row (sm_100a).
//
// Tensor-core path, one CTA per item (row tile x column chunk):
//   S[128 x 128] = X . W_tile^T     tcgen05.mma, TS form: A = the query tile X resident in TMEM (bf16 pairs, D/2 columns),
//                                   B = K-chunks [128 prototypes x 64 features] of queue_bf16[0] streamed by TMA (128-byte swizzle)
//   epilogue                        8 warps (2 warpgroups = 2 S accumulators, tiles alternate): tcgen05.ld S, chunk-max filter
//                                   against the row's k-th key, exact register top-k scan (topk_scan16, signed keys) of what passes
// This is the S-CTA of the training sweep without the exponentials, GEMM-2 and the O accumulator, so D = 512 fits one CTA (TMEM:
// X 256 columns + 2 x S 256) and no CTA pair is needed.  No W tile is read twice, so the ring holds 16 KB K-chunk stages.
// The column count is the LRU's device-side cur_idx (no host sync); each CTA derives its column range from it.  The chunks of a
// row share a threshold (kth_shared: atomicMax of every list's k-th key) so that a chunk skips what another chunk has beaten;
// entries whose key equals the shared value are kept (floor = shared - 1), which makes the union of the lists contain every key
// down to the row's k-th one whatever the timing.
//
// Check mode (fp32): one warp per (row, column chunk), fp64 dot products, the same lists.
// Both paths end in identify_merge_kernel: the k best keys of the row over all lists (ties: smaller slot), rescored as fp32 dots
// with fp64 accumulation against queue_f32[0], sorted by (score desc, slot asc), slot -> key through the LRU's slot_key[].
#include <cuda.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "identify_internal.cuh"
#include "sm100_ptx.cuh"

namespace ffc {
namespace idf {

constexpr int BM = 128;            // query rows per item
constexpr int BN = 128;            // prototypes per tile
constexpr int KC = 64;             // bf16 elements per 128-byte swizzle row
constexpr int NEPI = 2;            // epilogue warpgroups == S accumulators == top-k lists per item
constexpr int NTHREADS = 128 + NEPI * 128;
constexpr int STAGES = 12;         // K-chunk stages of the W ring
constexpr int STAGE_BYTES = BN * KC * 2;
constexpr int P_COL = 0, S_COL = 256;                                     // tensor-memory columns
constexpr size_t SMEM = 1024 + (size_t)STAGES * STAGE_BYTES + 1024;     // barriers, ring, alignment slack
constexpr int EMPTY_KEY = (int)0x80000000u;
constexpr int SIMT_WARPS = 8;
constexpr int MERGE_WARPS = 8;
static_assert(SMEM <= 227 * 1024, "shared memory budget");

struct Bars {
  uint64_t p_full;
  uint64_t full[STAGES];
  uint64_t empty[STAGES];
  uint64_t s_full[NEPI];
  uint64_t s_free[NEPI];
  uint32_t tmem_base;
};
static_assert(sizeof(Bars) <= 1024, "barrier block too large");

struct Params {
  const float* x;              // [n_rows, D] unit query rows (fp32)
  const float* w32;            // [q_local, D] queue_f32[0] (check mode)
  const int32_t* n_cols_dev;   // the LRU's cur_idx
  int64_t n_cols_max;          // q_local
  int n_rows, k, n_chunks, D;
  int32_t* kth_shared;         // [n_rows], INT_MIN-initialised (tensor-core path)
  int32_t* key_part;           // [n_lists][n_rows][k] descending keys, EMPTY_KEY padded
  int32_t* slot_part;          // [n_lists][n_rows][k] LOCAL slots or -1
};

__device__ __forceinline__ int64_t resident_cols(const Params& p) {
  const int64_t n = (int64_t)__ldcg(p.n_cols_dev);
  return n < 0 ? 0 : (n > p.n_cols_max ? p.n_cols_max : n);
}

// smallest float whose keys can exceed `kth` (keys drop the low 5 bits of topk_ord)
__device__ __forceinline__ float key_floor_value(int kth) {
  if (kth < topk_ord(0xff800000u)) return -INFINITY;
  const int kv = kth & (int)TOPK_VAL_MASK;
  return __uint_as_float(kv >= 0 ? (uint32_t)kv : ((uint32_t)kv ^ 0x7fffffffu));
}

template <int D>
__global__ void __launch_bounds__(NTHREADS, 1) ffc_identify_sm100_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ Params prm) {
  constexpr int NKC = D / KC;
  static_assert(P_COL + D / 2 <= S_COL && S_COL + NEPI * BN <= 512, "tensor memory budget");
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  Bars& bars = *reinterpret_cast<Bars*>(smem);
  unsigned char* sW = smem + 1024;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_row_tiles = (prm.n_rows + BM - 1) / BM;
  const int rt = blockIdx.x % n_row_tiles, chunk = blockIdx.x / n_row_tiles;
  const int row0 = rt * BM;
  const int64_t n_cols = resident_cols(prm);
  const int n_tiles_total = (int)((n_cols + BN - 1) / BN);
  const int tiles_per_chunk = (n_tiles_total + prm.n_chunks - 1) / prm.n_chunks;
  const int t_begin = min(chunk * tiles_per_chunk, n_tiles_total);
  const int t_end = min(t_begin + tiles_per_chunk, n_tiles_total);
  const int n_tiles = t_end - t_begin;

  if (threadIdx.x == 0) {
    mbar_init(&bars.p_full, 4);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&bars.full[i], 1);
      mbar_init(&bars.empty[i], 1);
    }
    for (int i = 0; i < NEPI; ++i) {
      mbar_init(&bars.s_full[i], 1);
      mbar_init(&bars.s_free[i], 4);
    }
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
    // ---- TMA producer: K-chunk [BN prototypes x 64 features] per stage ----
    int stage = 0;
    uint32_t ph = 0;
    for (int t = t_begin; t < t_end; ++t) {
      for (int kc = 0; kc < NKC; ++kc) {
        mbar_wait(&bars.empty[stage], ph ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&bars.full[stage], (uint32_t)STAGE_BYTES);
          tma_load_2d(&map_w, &bars.full[stage], sW + stage * STAGE_BYTES, kc * KC, t * BN);
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          ph ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // ---- MMA issue (converged warp, one elected lane): tile i into S buffer i & 1 once its epilogue has read it ----
    if (n_tiles > 0) {
      constexpr uint32_t idesc = make_idesc(BM, BN, 0, 0);
      mbar_wait(&bars.p_full, 0);
      tc_fence_after();
      const uint64_t b0 = make_desc(smem_u32(sW), 16, 1024);
      int stage = 0;
      uint32_t ph = 0;
      for (int i = 0; i < n_tiles; ++i) {
        const int buf = i & 1;
        mbar_wait(&bars.s_free[buf], (((uint32_t)i >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t tmem_s = tmem_base + (uint32_t)(S_COL + buf * BN);
        for (int kc = 0; kc < NKC; ++kc) {
          mbar_wait(&bars.full[stage], ph);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t bd = b0 + (uint64_t)((stage * STAGE_BYTES) >> 4);
            const uint32_t ta = tmem_base + (uint32_t)(P_COL + kc * (KC / 2));
#pragma unroll
            for (int k = 0; k < KC / 16; ++k) tc_mma_ts(tmem_s, ta + (uint32_t)(8 * k), bd + (uint64_t)(2 * k), idesc, (kc | k) ? 1u : 0u);
            tc_commit(&bars.empty[stage]);
            if (kc == NKC - 1) tc_commit(&bars.s_full[buf]);
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            ph ^= 1;
          }
        }
      }
    }
  } else if (warp >= 4) {
    // ---- epilogue: warpgroup g takes the tiles of parity g ----
    const int g = (warp - 4) >> 2;
    const int q4 = warp & 3;                    // TMEM lane quarter
    const int row = row0 + q4 * 32 + lane;
    const bool row_ok = row < prm.n_rows;
    const int k = prm.k;
    int tk[KMAX], tc[KMAX];
#pragma unroll
    for (int q = 0; q < KMAX; ++q) {
      tk[q] = EMPTY_KEY;
      tc[q] = -1;
    }
    int kth = EMPTY_KEY, kfloor = EMPTY_KEY, kpub = EMPTY_KEY;
    int32_t* kshare = row_ok ? prm.kth_shared + row : nullptr;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16);
    if (g == 0 && n_tiles > 0) {
      // query tile -> TMEM (the A operand of every MMA of this item): thread = row, fp32 -> bf16 pairs, 32 columns per store
      const float4* src = reinterpret_cast<const float4*>(prm.x + (int64_t)(row_ok ? row : 0) * D);
#pragma unroll 1
      for (int c0 = 0; c0 < D / 2; c0 += 32) {
        uint32_t v[32];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          const float4 t = row_ok ? __ldg(src + c0 / 2 + q) : make_float4(0.f, 0.f, 0.f, 0.f);
          v[2 * q] = pack_bf16(t.x, t.y);
          v[2 * q + 1] = pack_bf16(t.z, t.w);
        }
        tc_st32(lane_base + (uint32_t)(P_COL + c0), v);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.p_full);
    }
    uint32_t use = 0;
    for (int i = g; i < n_tiles; i += NEPI, ++use) {
      const int64_t j0 = (int64_t)(t_begin + i) * BN;
      if (kshare) {
        const int ks = __ldcg(kshare);
        if (ks != EMPTY_KEY) kfloor = max(kfloor, ks - 1);
      }
      kth = max(kth, kfloor);
      float thrf = key_floor_value(kth);
      mbar_wait(&bars.s_full[g], use & 1);
      tc_fence_after();
      const uint32_t tmem_s = lane_base + (uint32_t)(S_COL + g * BN);
#pragma unroll 1
      for (int cc = 0; cc < BN / 32; ++cc) {
        uint32_t v[32];
        tc_ld32(tmem_s + cc * 32, v);
        const int col0 = (int)j0 + cc * 32;
        uint32_t excl = 0u;
        if ((int64_t)col0 + 32 > n_cols) {
          const int nv = (int)(n_cols - col0);
          excl = nv <= 0 ? 0xffffffffu : (0xffffffffu << nv);
        }
        float m0 = __uint_as_float(v[0]), m1 = __uint_as_float(v[1]);
#pragma unroll
        for (int c = 2; c < 32; c += 2) {
          m0 = fmaxf(m0, __uint_as_float(v[c]));
          m1 = fmaxf(m1, __uint_as_float(v[c + 1]));
        }
        if (__any_sync(0xffffffffu, row_ok && fmaxf(m0, m1) >= thrf)) {
          topk_scan16<0, 32, true>(v, excl & 0xffffu, col0, row_ok, k, tk, tc, kth, kfloor);
          topk_scan16<16, 32, true>(v, excl >> 16, col0 + 16, row_ok, k, tk, tc, kth, kfloor);
          thrf = key_floor_value(kth);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.s_free[g]);
      if (kshare) {
        int kown = EMPTY_KEY;
#pragma unroll
        for (int r = 0; r < KMAX; ++r)
          if (r == k - 1) kown = tk[r];
        if (kown > kpub) {
          atomicMax(kshare, kown);
          kpub = kown;
        }
      }
    }
    if (row_ok) {
      const int64_t base = ((int64_t)(chunk * NEPI + g) * prm.n_rows + row) * k;
#pragma unroll
      for (int q = 0; q < KMAX; ++q) {
        if (q < k) {
          prm.key_part[base + q] = tk[q];
          prm.slot_part[base + q] = tc[q] >= 0 ? tc[q] + (tk[q] & 31) : -1;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
}

// fp32 result of the fp64-accumulated dot of two fp32 rows (D a multiple of 4); every lane of the warp returns the same bits
__device__ __forceinline__ float warp_dot(const float* __restrict__ a, const float* __restrict__ b, int D, int lane) {
  double s = 0.0;
  for (int e = lane * 4; e < D; e += 128) {
    const float4 x = *reinterpret_cast<const float4*>(a + e);
    const float4 y = __ldg(reinterpret_cast<const float4*>(b + e));
    s = fma((double)x.x, (double)y.x, s);
    s = fma((double)x.y, (double)y.y, s);
    s = fma((double)x.z, (double)y.z, s);
    s = fma((double)x.w, (double)y.w, s);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  return (float)s;
}

// check mode: warp = (row, column chunk); the list is warp-uniform, columns ascending, so equal keys keep the smaller slot
__global__ void __launch_bounds__(SIMT_WARPS * 32) ffc_identify_simt_kernel(const Params prm) {
  const int lane = threadIdx.x & 31;
  const int64_t item = (int64_t)blockIdx.x * SIMT_WARPS + (threadIdx.x >> 5);
  if (item >= (int64_t)prm.n_rows * prm.n_chunks) return;
  const int row = (int)(item % prm.n_rows), chunk = (int)(item / prm.n_rows);
  const int D = prm.D, k = prm.k;
  const int64_t n_cols = resident_cols(prm);
  const int64_t per = (n_cols + prm.n_chunks - 1) / prm.n_chunks;
  const int64_t c_begin = std::min<int64_t>(chunk * per, n_cols), c_end = std::min<int64_t>(c_begin + per, n_cols);
  const float* x = prm.x + (int64_t)row * D;
  int tk[KMAX], ts[KMAX];
#pragma unroll
  for (int q = 0; q < KMAX; ++q) {
    tk[q] = EMPTY_KEY;
    ts[q] = -1;
  }
  int kth = EMPTY_KEY;
  for (int64_t j = c_begin; j < c_end; ++j) {
    const int key = topk_ord(__float_as_uint(warp_dot(x, prm.w32 + j * D, D, lane)));
    if (key > kth) {
      topk_insert_key(key, (int)j, k, tk, ts);
#pragma unroll
      for (int r = 0; r < KMAX; ++r)
        if (r == k - 1) kth = tk[r];
    }
  }
  if (lane == 0) {
    const int64_t base = ((int64_t)chunk * prm.n_rows + row) * k;
#pragma unroll
    for (int q = 0; q < KMAX; ++q) {
      if (q < k) {
        prm.key_part[base + q] = tk[q];
        prm.slot_part[base + q] = ts[q];
      }
    }
  }
}

__device__ __forceinline__ bool ranks_before(int ka, int sa, int kb, int sb) { return ka > kb || (ka == kb && sa < sb); }

// merge: warp = row.  Each lane keeps the best k of a strided share of the row's candidates; k rounds of a warp arg-max pick the
// winners; they are rescored, sorted by (score desc, slot asc) and written with their labels.  Missing entries: slot -1,
// label INT64_MIN, score -inf.
__global__ void __launch_bounds__(MERGE_WARPS * 32) ffc_identify_merge_kernel(const Params prm, int n_lists, const int64_t* __restrict__ slot_key,
                                                                            int64_t col_offset, float* __restrict__ score_out,
                                                                            int64_t* __restrict__ label_out, int32_t* __restrict__ slot_out) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * MERGE_WARPS + (threadIdx.x >> 5);
  if (row >= prm.n_rows) return;
  const int k = prm.k, D = prm.D;
  constexpr int NONE = 0x7fffffff;
  int lk[KMAX], ls[KMAX];
#pragma unroll
  for (int q = 0; q < KMAX; ++q) {
    lk[q] = EMPTY_KEY;
    ls[q] = NONE;
  }
  const int n_cand = n_lists * k;
  for (int e = lane; e < n_cand; e += 32) {
    const int64_t idx = ((int64_t)(e / k) * prm.n_rows + row) * k + e % k;
    int xs = prm.slot_part[idx];
    if (xs < 0) continue;
    int xk = prm.key_part[idx];
#pragma unroll
    for (int r = 0; r < KMAX; ++r) {
      if (r < k && ranks_before(xk, xs, lk[r], ls[r])) {
        const int tk = lk[r], ts = ls[r];
        lk[r] = xk;
        ls[r] = xs;
        xk = tk;
        xs = ts;
      }
    }
  }
  int ws[KMAX];
  float sc[KMAX];
#pragma unroll
  for (int r = 0; r < KMAX; ++r) {
    ws[r] = -1;
    sc[r] = -INFINITY;
    if (r < k) {
      int bk = lk[0], bs = ls[0];
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        const int ok = __shfl_xor_sync(0xffffffffu, bk, o), os = __shfl_xor_sync(0xffffffffu, bs, o);
        if (ranks_before(ok, os, bk, bs)) {
          bk = ok;
          bs = os;
        }
      }
      if (bs != NONE) {
        if (ls[0] == bs) {      // slots are unique: exactly one lane holds the winner at its head
#pragma unroll
          for (int q = 0; q + 1 < KMAX; ++q) {
            lk[q] = lk[q + 1];
            ls[q] = ls[q + 1];
          }
          lk[KMAX - 1] = EMPTY_KEY;
          ls[KMAX - 1] = NONE;
        }
        ws[r] = bs;
        sc[r] = warp_dot(prm.x + (int64_t)row * D, prm.w32 + (int64_t)bs * D, D, lane);
      }
    }
  }
  if (lane == 0) {
    // selection sort of the (at most KMAX) winners by (score desc, slot asc); missing entries stay last
#pragma unroll
    for (int a = 0; a < KMAX; ++a) {
#pragma unroll
      for (int b = a + 1; b < KMAX; ++b) {
        const bool swap = ws[b] >= 0 && (ws[a] < 0 || sc[b] > sc[a] || (sc[b] == sc[a] && ws[b] < ws[a]));
        if (swap) {
          const float tsc = sc[a];
          const int tsl = ws[a];
          sc[a] = sc[b];
          ws[a] = ws[b];
          sc[b] = tsc;
          ws[b] = tsl;
        }
      }
    }
#pragma unroll
    for (int q = 0; q < KMAX; ++q) {
      if (q < k) {
        const int64_t o = (int64_t)row * k + q;
        const bool live = ws[q] >= 0;
        score_out[o] = live ? sc[q] : -INFINITY;
        slot_out[o] = live ? (int32_t)(col_offset + ws[q]) : -1;
        label_out[o] = live ? slot_key[ws[q]] : INT64_MIN;
      }
    }
  }
}

template <int D>
static int launch_tc(const CUtensorMap& map, const Params& p, int n_items, cudaStream_t s) {
  static bool attr_set = false;
  auto kern = ffc_identify_sm100_kernel<D>;
  if (!attr_set) {
    FFC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
    attr_set = true;
  }
  kern<<<dim3(n_items), dim3(NTHREADS), SMEM, s>>>(map, p);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

static int64_t align256(int64_t b) { return (b + 255) / 256 * 256; }

}  // namespace idf

// Column chunks per row: one wave of 148 items (tensor-core path: 148 CTAs, one per SM; check mode: 32 warps per SM), never more
// chunks than there can be tiles (columns) in the queue.
int identify_chunks(bool bf16, int n_rows, int64_t q_local) {
  if (bf16) {
    const int row_tiles = (n_rows + idf::BM - 1) / idf::BM;
    return (int)std::max<int64_t>(1, std::min<int64_t>(148 / row_tiles, ceil_div64(q_local, idf::BN)));
  }
  return (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(148 * 32 / n_rows, 256), q_local));
}

int identify_lists(bool bf16, int n_rows, int64_t q_local) { return identify_chunks(bf16, n_rows, q_local) * (bf16 ? idf::NEPI : 1); }

int64_t identify_workspace_bytes(bool bf16, int n_rows, int k, int64_t q_local) {
  const int64_t part = idf::align256((int64_t)identify_lists(bf16, n_rows, q_local) * n_rows * k * 4);
  return idf::align256((int64_t)n_rows * 4) + 2 * part;
}

int launch_identify(Sm100Cache* cache, const IdentifyArgs& a, cudaStream_t s) {
  const bool bf16 = a.queue_bf16 != nullptr;
  idf::Params p;
  memset(&p, 0, sizeof(p));
  p.x = a.x;
  p.w32 = a.queue_f32;
  p.n_cols_dev = a.cur_idx_dev;
  p.n_cols_max = a.q_local;
  p.n_rows = a.n_rows;
  p.k = a.k;
  p.D = a.D;
  p.n_chunks = identify_chunks(bf16, a.n_rows, a.q_local);
  const int n_lists = identify_lists(bf16, a.n_rows, a.q_local);
  char* ws = static_cast<char*>(a.workspace);
  const int64_t part = idf::align256((int64_t)n_lists * a.n_rows * a.k * 4);
  p.kth_shared = reinterpret_cast<int32_t*>(ws);
  p.key_part = reinterpret_cast<int32_t*>(ws + idf::align256((int64_t)a.n_rows * 4));
  p.slot_part = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(p.key_part) + part);
  if (bf16) {
    CUtensorMap map;
    int rc = sm100_get_map(cache, a.queue_bf16, a.q_local, a.D, idf::BN, false, &map);
    if (rc) return rc;
    FFC_CUDA(cudaMemsetAsync(p.kth_shared, 0x80, (size_t)a.n_rows * 4, s));    // 0x80808080: below every key of a cosine
    const int n_items = ((a.n_rows + idf::BM - 1) / idf::BM) * p.n_chunks;
    switch (a.D) {
      case 64: rc = idf::launch_tc<64>(map, p, n_items, s); break;
      case 128: rc = idf::launch_tc<128>(map, p, n_items, s); break;
      case 256: rc = idf::launch_tc<256>(map, p, n_items, s); break;
      case 512: rc = idf::launch_tc<512>(map, p, n_items, s); break;
      default: FFC_REQUIRE(false, "ffc_identify: the bf16 path is built for D 64, 128, 256 or 512 (got %d)", a.D);
    }
    if (rc) return rc;
  } else {
    const int64_t warps = (int64_t)a.n_rows * p.n_chunks;
    idf::ffc_identify_simt_kernel<<<(unsigned)((warps + idf::SIMT_WARPS - 1) / idf::SIMT_WARPS), idf::SIMT_WARPS * 32, 0, s>>>(p);
    FFC_LAUNCH_CHECK();
  }
  idf::ffc_identify_merge_kernel<<<(a.n_rows + idf::MERGE_WARPS - 1) / idf::MERGE_WARPS, idf::MERGE_WARPS * 32, 0, s>>>(
      p, n_lists, a.slot_key, a.col_offset, a.score_out, a.label_out, a.slot_out);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

}  // namespace ffc
