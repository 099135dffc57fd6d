// Fused margin-softmax head: handle, prep, check-mode (fp32 in / fp64 accumulate, SIMT) sweep,
// partial reduce and finalize.  Replaces ffc.py:195-202 / 248-254 + add_margin (ffc.py:60-138) and
// its autograd backward.  The tcgen05 sweep lives in head_sm100.cu and produces the same partials.
//
// Math (per probe row i, loss l in {1,2}; s = scale, M = fixed max, f = margin function):
//   p~_ij = exp(s*z_ij - M) over all columns j except the target t_i and the `ones` set C
//   L_l   = sum_common p~ + sum_{j in C\{t}} p~(W_l[j]) + exp(s*f(cos_t,l) - M)
//   CE_l  = log L_l + M - s*f(cos_t,l)                                  (F.cross_entropy, ffc.py:83/104/127)
//   dCE_l/dp = s * [ (O_common + O_side,l)/L_l + (e_t/L_l - 1) * f'(cos_t,l) * W_l[t] ]
// with W_1 = queue[0], W_2 = queue[1] on C and queue[0] elsewhere (ffc.py:197-200), O = sum p~_j W_j.
// Hard negatives (ffc.py:86-92): mean over outlier rows and their top-k cosines of max(cos, 0).
#include <algorithm>
#include <math.h>
#include <vector>

#include "identify_internal.cuh"

namespace ffc {
struct ReduceJobs;
}

struct ffc_head {
  ffc_head_config cfg;
  int64_t part_rows_cap;
  int max_chunks;
  // workspace
  __nv_bfloat16* p16;
  float* side_f32;             // [2][max_rows][D]
  __nv_bfloat16* side_bf16;    // [2][max_rows][D]
  int32_t* tcol;               // [max_rows]  target column in the main sweep (local) or -1
  int32_t* tpos;               // [max_rows]  target position in ones_list or -1
  uint8_t* is_out;             // [max_rows]
  int32_t* kth_shared;         // [max_rows] hard-negative threshold shared by the column chunks of the tcgen05 sweep
  float* thr;                  // [2][max_rows]
  int32_t* counts;             // [2][2] n_pos, n_out, double-buffered by pass parity
  int32_t* row_map;            // [max_rows] sweep position -> probe row: positives first, hard-negative-only rows last (prep kernel's last block)
  int32_t* part_ctr;           // [2]: arrival counter of the prep blocks, number of rows in front of the hard-negative-only rows
  int pass_parity;
  int prepared_rows;           // rows of the last ffc_head_prep not yet swept (ffc_head_prep / ffc_head_sweep_prepared pairing), else <= 0
  ffc::ReduceJobs* jobs;        // partial-result descriptors of the last merged sweep launch (one-GPU fast path)
  int jobs_pending;            // 1: the last sweep left its partials unreduced for head_finalize_fused_kernel
  float* row_loss;             // [max_rows]
  float* coef;                 // [4][max_rows] finalize coefficients
  int32_t* nslot;              // [max_rows] hard-negative gather count
  int32_t* wslot;              // [max_rows][2*KMAX]
  uint8_t* wrow;               // [max_rows][2*KMAX]
  float* l_part;
  float* o_part;
  float* topv_part;
  int32_t* topi_part;
  ffc::Sm100Cache* sm100;
  // queue-gradient mode (ffc_head_set_dqueue / ffc_head_dqueue)
  int want_dq;
  __nv_bfloat16* pc16;         // [max_rows][D] probe rows scaled by their softmax coefficients (GEMM-2 operand of the swapped sweep; bf16 AM / Arc)
  float4* dq_col;              // [max_rows] (thr_1, thr_2, a_1, a_2) per probe row: the column scalars of the swapped SV sweep (bf16 SV)
  float* dq_l;                 // [q_local] scratch partials of the swapped sweep (denominators: unused)
  float* dq_tv;                // [q_local]
  int32_t* dq_ti;              // [q_local]
  int32_t* dq_claim;           // [q_local] which call last claimed a special slot
  int32_t dq_epoch;
  // optional device timing of the main sweep kernel (bench / roofline evidence)
  int timing;
  std::vector<cudaEvent_t>* ev;   // pairs (start, stop), recorded on the launch stream
  size_t ev_used;
};

namespace ffc {

// ------------------------------------------------------------------------------------------------
// prep
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) head_prep_rows_kernel(const int32_t* __restrict__ label, int n_rows, int64_t col_offset, int64_t q_local,
                                                             const uint32_t* __restrict__ cmask, const int32_t* __restrict__ ones_list,
                                                             const int32_t* __restrict__ n_ones_p, int32_t* __restrict__ tcol,
                                                             int32_t* __restrict__ tpos, uint8_t* __restrict__ is_out, int32_t* counts) {
  // one block per row so that the ones_list search is parallel
  const int i = blockIdx.x;
  const int32_t lab = label[i];
  int32_t tc = -1;
  if (lab >= 0) {
    const int64_t loc = (int64_t)lab - col_offset;
    if (loc >= 0 && loc < q_local) tc = (int32_t)loc;
  }
  __shared__ int found;
  if (threadIdx.x == 0) found = -1;
  __syncthreads();
  const bool in_c = (tc >= 0) && cmask && ((cmask[tc >> 5] >> (tc & 31)) & 1u);
  if (in_c) {
    const int no = *n_ones_p;
    for (int j = threadIdx.x; j < no; j += blockDim.x)
      if (ones_list[j] == tc) found = j;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    tcol[i] = tc;
    tpos[i] = found;
    is_out[i] = lab < 0;
    atomicAdd(&counts[lab < 0 ? 1 : 0], 1);
  }
}

// side matrices: W_side0[j] = queue[0][ones[j]], W_side1[j] = queue[1][ones[j]]
__global__ void __launch_bounds__(128) head_gather_side_kernel(const float* __restrict__ qf, const __nv_bfloat16* __restrict__ qh, int64_t q_local, int D,
                                                               const int32_t* __restrict__ ones_list, const int32_t* __restrict__ n_ones_p,
                                                               int max_rows, float* __restrict__ side_f32, __nv_bfloat16* __restrict__ side_bf16) {
  const int j = blockIdx.x;
  const int no = *n_ones_p;
  if (j >= ((no + 127) & ~127)) return;   // only the tiles the side sweeps will touch need rows (zero padded to 128)
  const bool live = j < no;
  const int64_t slot = live ? ones_list[j] : 0;
  for (int r = 0; r < 2; ++r) {
    const int64_t src = ((int64_t)r * q_local + slot) * D;
    const int64_t dst = ((int64_t)r * max_rows + j) * D;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
      if (side_f32) side_f32[dst + d] = live ? qf[src + d] : 0.f;
      if (side_bf16) side_bf16[dst + d] = live ? qh[src + d] : __float2bfloat16(0.f);
    }
  }
}

// target cosines: tgt[0] = p . queue[0][t], tgt[1] = p . (t in C ? queue[1][t] : queue[0][t]), tgt[2] = owner
template <bool BF16>
__global__ void __launch_bounds__(128) head_target_kernel(const float* __restrict__ P, const __nv_bfloat16* __restrict__ P16, const float* __restrict__ qf,
                                                          const __nv_bfloat16* __restrict__ qh, int64_t q_local, int D, int n_rows,
                                                          const int32_t* __restrict__ tcol, const int32_t* __restrict__ tpos, float margin,
                                                          float* __restrict__ tgt, float* __restrict__ thr) {
  const int i = blockIdx.x;
  const int32_t tc = tcol[i];
  double a0 = 0.0, a1 = 0.0;
  if (tc >= 0) {
    const int64_t r0 = (int64_t)tc * D;
    const int64_t r1 = (tpos[i] >= 0) ? ((int64_t)q_local + tc) * D : r0;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
      float p, w0, w1;
      if (BF16) {
        p = __bfloat162float(P16[(int64_t)i * D + d]);
        w0 = __bfloat162float(qh[r0 + d]);
        w1 = __bfloat162float(qh[r1 + d]);
      } else {
        p = P[(int64_t)i * D + d];
        w0 = qf[r0 + d];
        w1 = qf[r1 + d];
      }
      a0 += (double)p * w0;
      a1 += (double)p * w1;
    }
  }
  __shared__ double s0[128], s1[128];
  s0[threadIdx.x] = a0;
  s1[threadIdx.x] = a1;
  __syncthreads();
  for (int o = 64; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      s0[threadIdx.x] += s0[threadIdx.x + o];
      s1[threadIdx.x] += s1[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const float c0 = (float)s0[0], c1 = (float)s1[0];
    tgt[0 * n_rows + i] = tc >= 0 ? c0 : 0.f;
    tgt[1 * n_rows + i] = tc >= 0 ? c1 : 0.f;
    tgt[2 * n_rows + i] = tc >= 0 ? 1.f : 0.f;
    tgt[3 * n_rows + i] = 0.f;
    if (thr) {
      thr[i] = tc >= 0 ? c0 - margin : INFINITY;
      thr[n_rows + i] = tc >= 0 ? c1 - margin : INFINITY;
    }
  }
}

// Everything a pass needs before its sweep, in ONE launch (block b: probe row b and/or side row b):
//   row part   (b < n_rows): target column / position in `ones` / outlier flag / n_pos, n_out counts (head_prep_rows_kernel),
//                            bf16 copy of the probe row (head_p_to_bf16_kernel), target cosines (head_target_kernel)
//   side part  (b < ceil128(n_ones)): gathered `ones` rows of queue[0] and queue[1] (head_gather_side_kernel)
// counts[2][2] is double-buffered by pass parity: block 0 clears the other parity's pair for the next pass (no memset launch).
template <bool BF16>
__global__ void __launch_bounds__(128) head_prep_fused_kernel(const float* __restrict__ P, __nv_bfloat16* __restrict__ P16, const int32_t* __restrict__ label,
                                                              int n_rows, int64_t col_offset, int64_t q_local, int D, const float* __restrict__ qf,
                                                              const __nv_bfloat16* __restrict__ qh, const uint32_t* __restrict__ cmask,
                                                              const int32_t* __restrict__ ones_list, const int32_t* __restrict__ n_ones_p, int max_rows,
                                                              float* __restrict__ side_f32, __nv_bfloat16* __restrict__ side_bf16,
                                                              int32_t* __restrict__ tcol, int32_t* __restrict__ tpos, uint8_t* __restrict__ is_out,
                                                              int32_t* __restrict__ kth_shared, int32_t* counts_cur, int32_t* counts_next, float margin,
                                                              float* __restrict__ tgt, float* __restrict__ thr, int32_t* __restrict__ row_map,
                                                              int32_t* part_ctr) {
  const int b = blockIdx.x;
  const int no = *n_ones_p;
  __shared__ int found;
  __shared__ double s0[128], s1[128];
  if (b == 0 && threadIdx.x < 2) counts_next[threadIdx.x] = 0;
  if (b < n_rows) {
    const int i = b;
    const int32_t lab = label[i];
    int32_t tc = -1;
    if (lab >= 0) {
      const int64_t loc = (int64_t)lab - col_offset;
      if (loc >= 0 && loc < q_local) tc = (int32_t)loc;
    }
    if (threadIdx.x == 0) found = -1;
    __syncthreads();
    const bool in_c = (tc >= 0) && cmask && ((cmask[tc >> 5] >> (tc & 31)) & 1u);
    if (in_c) {
      for (int j = threadIdx.x; j < no; j += blockDim.x)
        if (ones_list[j] == tc) found = j;
    }
    __syncthreads();
    const int fpos = found;
    if (threadIdx.x == 0) {
      tcol[i] = tc;
      tpos[i] = fpos;
      is_out[i] = lab < 0;
      kth_shared[i] = 0;
      atomicAdd(&counts_cur[lab < 0 ? 1 : 0], 1);
    }
    // bf16 probe row + target cosines: tgt[0] = p . queue[0][t], tgt[1] = p . (t in C ? queue[1][t] : queue[0][t])
    double a0 = 0.0, a1 = 0.0;
    const int64_t r0 = (int64_t)(tc >= 0 ? tc : 0) * D;
    const int64_t r1 = (fpos >= 0) ? ((int64_t)q_local + tc) * D : r0;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
      float p = P[(int64_t)i * D + d];
      if (BF16) {
        const __nv_bfloat16 pb = __float2bfloat16(p);
        P16[(int64_t)i * D + d] = pb;
        p = __bfloat162float(pb);
      }
      if (tc >= 0) {
        const float w0 = BF16 ? __bfloat162float(qh[r0 + d]) : qf[r0 + d];
        const float w1 = BF16 ? __bfloat162float(qh[r1 + d]) : qf[r1 + d];
        a0 += (double)p * w0;
        a1 += (double)p * w1;
      }
    }
    s0[threadIdx.x] = a0;
    s1[threadIdx.x] = a1;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
      if (threadIdx.x < o) {
        s0[threadIdx.x] += s0[threadIdx.x + o];
        s1[threadIdx.x] += s1[threadIdx.x + o];
      }
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      const float c0 = (float)s0[0], c1 = (float)s1[0];
      tgt[0 * n_rows + i] = tc >= 0 ? c0 : 0.f;
      tgt[1 * n_rows + i] = tc >= 0 ? c1 : 0.f;
      tgt[2 * n_rows + i] = tc >= 0 ? 1.f : 0.f;
      tgt[3 * n_rows + i] = 0.f;
      if (thr) {
        thr[i] = tc >= 0 ? c0 - margin : INFINITY;
        thr[n_rows + i] = tc >= 0 ? c1 - margin : INFINITY;
      }
    }
  }
  // side matrices: W_side0[j] = queue[0][ones[j]], W_side1[j] = queue[1][ones[j]], zero padded to the 128-row tile
  if (b < ((no + 127) & ~127) && b < max_rows) {
    const int j = b;
    const bool live = j < no;
    const int64_t slot = live ? ones_list[j] : 0;
    for (int r = 0; r < 2; ++r) {
      const int64_t src = ((int64_t)r * q_local + slot) * D;
      const int64_t dst = ((int64_t)r * max_rows + j) * D;
      for (int d = threadIdx.x; d < D; d += blockDim.x) {
        if (side_f32) side_f32[dst + d] = live ? qf[src + d] : 0.f;
        if (side_bf16) side_bf16[dst + d] = live ? qh[src + d] : __float2bfloat16(0.f);
      }
    }
  }
  // Row order of the tcgen05 sweep: the last block to arrive writes the stable partition "rows with a softmax term first, hard-negative-
  // only rows (label -1, ffc.py:61) last" -- row tiles made of the latter need neither exponentials nor the second GEMM -- and the
  // number of rows in front.  At the very-large-scale end (C4: ten identities per queue slot) nine rows in ten are of that kind.
  if (row_map) {
    __shared__ int s_last;
    __shared__ int s_cnt[128];
    __threadfence();                    // this block's is_out[] is visible before its arrival is
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(part_ctr, 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (s_last) {
      __threadfence();
      const volatile uint8_t* vo = is_out;
      const int per = (n_rows + 127) / 128, r_begin = min(n_rows, (int)threadIdx.x * per), r_end = min(n_rows, r_begin + per);
      int np = 0;
      for (int i = r_begin; i < r_end; ++i) np += vo[i] ? 0 : 1;
      s_cnt[threadIdx.x] = np;
      __syncthreads();
      int before = 0, total = 0;
      for (int t = 0; t < 128; ++t) {
        const int c = s_cnt[t];
        if (t < (int)threadIdx.x) before += c;
        total += c;
      }
      int wp = before, wo = total + (r_begin - before);      // next free position among the positives / the hard-negative-only rows
      for (int i = r_begin; i < r_end; ++i) {
        if (vo[i]) row_map[wo++] = i;
        else row_map[wp++] = i;
      }
      if (threadIdx.x == 0) {
        part_ctr[1] = total;
        part_ctr[0] = 0;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// check-mode sweep: fp32 inputs, fp64 arithmetic, no tensor cores.  Block = 256 threads,
// 16 probe rows x one column chunk, 32 columns per step.
// ------------------------------------------------------------------------------------------------
constexpr int SR = 16;   // rows per block
constexpr int SC = 32;   // columns per step

__global__ void __launch_bounds__(256) head_sweep_simt_kernel(const SweepArgs a, int64_t cols_per_chunk) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int D = a.D;
  float* sP = reinterpret_cast<float*>(smem_raw);                  // [SR][D]
  float* sW = sP + SR * D;                                         // [SC][D]
  double* sG = reinterpret_cast<double*>(sW + SC * D);             // [SR][SC]  cos, then g~
  double* sL = sG + SR * SC;                                       // [SR]
  float* sTv = reinterpret_cast<float*>(sL + SR);                  // [SR][KMAX]
  int32_t* sTi = reinterpret_cast<int32_t*>(sTv + SR * KMAX);      // [SR][KMAX]

  const int tid = threadIdx.x;
  const int row0 = blockIdx.x * SR;
  const int chunk = blockIdx.y;
  const int64_t n_cols = a.n_cols_dev ? (int64_t)*a.n_cols_dev : a.n_cols;
  const int64_t c_begin = (int64_t)chunk * cols_per_chunk;
  int64_t c_end = c_begin + cols_per_chunk;
  if (c_end > n_cols) c_end = n_cols;

  for (int e = tid; e < SR * D; e += 256) {
    const int r = e / D, d = e - r * D;
    sP[e] = (row0 + r < a.n_rows) ? a.P_f32[(int64_t)(row0 + r) * D + d] : 0.f;
  }
  if (tid < SR) {
    sL[tid] = 0.0;
    for (int q = 0; q < KMAX; ++q) {
      sTv[tid * KMAX + q] = -INFINITY;
      sTi[tid * KMAX + q] = -1;
    }
  }
  const int orow = tid >> 4, od0 = tid & 15;   // O accumulation mapping: row, d = od0 + 16*q
  double acc[32];
#pragma unroll
  for (int q = 0; q < 32; ++q) acc[q] = 0.0;
  const double s = a.scale, M = a.fixed_max;
  __syncthreads();

  for (int64_t c0 = c_begin; c0 < c_end; c0 += SC) {
    const int nc = (int)((c_end - c0 < SC) ? (c_end - c0) : SC);
    for (int e = tid; e < SC * D; e += 256) {
      const int c = e / D, d = e - c * D;
      sW[e] = (c < nc) ? a.W_f32[(c0 + c) * D + d] : 0.f;
    }
    __syncthreads();
    // phase A: 16 x 32 cosines, two per thread
    for (int e = tid; e < SR * SC; e += 256) {
      const int r = e / SC, c = e - r * SC;
      double dot = 0.0;
      const float* pr = sP + r * D;
      const float* wc = sW + c * D;
      for (int d = 0; d < D; ++d) dot += (double)pr[d] * (double)wc[d];
      sG[e] = dot;
    }
    __syncthreads();
    // phase B: one thread per row: exclusions, exp, denominator, top-k
    if (tid < SR) {
      const int r = tid, gr = row0 + r;
      if (gr < a.n_rows) {
        const int32_t tc = a.tcol[gr];
        const double th = a.thr ? (double)a.thr[gr] : (double)INFINITY;
        const bool outl = a.is_out[gr];
        float tv[KMAX];
        int32_t ti[KMAX];
        for (int q = 0; q < KMAX; ++q) {
          tv[q] = sTv[r * KMAX + q];
          ti[q] = sTi[r * KMAX + q];
        }
        double lsum = 0.0;
        for (int c = 0; c < SC; ++c) {
          const int64_t col = c0 + c;
          bool excl = (c >= nc) || (col == tc);
          if (!excl && a.cmask) excl = (a.cmask[col >> 5] >> (col & 31)) & 1u;
          double g = 0.0;
          if (!excl) {
            const double cs = sG[r * SC + c];
            double z = cs, coef = 1.0;
            if (a.sv && cs > th) {
              z = (double)SV_T * cs + (double)SV_T - 1.0;
              coef = (double)SV_T;
            }
            const double pt = exp(s * z - M);
            lsum += pt;
            g = pt * coef;
            if (outl && (float)cs > tv[a.k - 1]) topk_insert<KMAX>(tv, ti, a.k, (float)cs, (int32_t)col);
          }
          sG[r * SC + c] = g;
        }
        sL[r] += lsum;
        for (int q = 0; q < KMAX; ++q) {
          sTv[r * KMAX + q] = tv[q];
          sTi[r * KMAX + q] = ti[q];
        }
      } else {
        for (int c = 0; c < SC; ++c) sG[r * SC + c] = 0.0;
      }
    }
    __syncthreads();
    // phase C: O[r][d] += g~[r][c] * W[c][d]
    for (int c = 0; c < nc; ++c) {
      const double g = sG[orow * SC + c];
      if (g != 0.0) {
        const float* wc = sW + c * D;
#pragma unroll
        for (int q = 0; q < 32; ++q) {
          const int d = od0 + 16 * q;
          if (d < D) acc[q] += g * (double)wc[d];
        }
      }
    }
    __syncthreads();
  }
  // write partials
  const int gr = row0 + orow;
  if (gr < a.n_rows) {
    float* op = a.o_part + ((int64_t)chunk * a.n_rows + gr) * D;
#pragma unroll
    for (int q = 0; q < 32; ++q) {
      const int d = od0 + 16 * q;
      if (d < D) op[d] = (float)acc[q];
    }
  }
  if (tid < SR && row0 + tid < a.n_rows) {
    const int64_t pr = (int64_t)chunk * a.n_rows + row0 + tid;
    a.l_part[pr] = (float)sL[tid];
    for (int q = 0; q < a.k; ++q) {
      a.topv_part[pr * a.k + q] = sTv[tid * KMAX + q];
      a.topi_part[pr * a.k + q] = sTi[tid * KMAX + q];
    }
  }
}

int launch_sweep_simt(const SweepArgs& a, cudaStream_t s) {
  FFC_REQUIRE(a.D <= 512, "check-mode sweep: D=%d > 512", a.D);
  const int row_tiles = (a.n_rows + SR - 1) / SR;
  const int64_t cpc = ((ceil_div64(a.n_cols, a.n_chunks) + SC - 1) / SC) * SC;
  const size_t smem = (size_t)(SR + SC) * a.D * sizeof(float) + (SR * SC + SR) * sizeof(double) + SR * KMAX * 8;
  static bool attr_set = false;
  if (!attr_set) {
    FFC_CUDA(cudaFuncSetAttribute(head_sweep_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    attr_set = true;
  }
  dim3 grid(row_tiles, a.n_chunks);
  head_sweep_simt_kernel<<<grid, 256, smem, s>>>(a, cpc);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

static int simt_pick_chunks(int n_rows, int64_t n_cols) {
  const int row_tiles = (n_rows + SR - 1) / SR;
  int64_t c = (4 * 148) / std::max(row_tiles, 1);
  c = std::min<int64_t>(c, ceil_div64(n_cols, SC));
  return (int)std::max<int64_t>(c, 1);
}

// ------------------------------------------------------------------------------------------------
// reduce partials over chunks -> stats slot `slot` (lsum/osum) and top-k slot `tslot` (or -1)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) head_reduce_kernel(const float* __restrict__ l_part, const float* __restrict__ o_part,
                                                          const float* __restrict__ topv_part, const int32_t* __restrict__ topi_part, int n_chunks,
                                                          int n_rows, int D, int k, float* __restrict__ lsum, float* __restrict__ osum,
                                                          float* __restrict__ topv, int32_t* __restrict__ topi, const uint8_t* __restrict__ is_out,
                                                          int64_t idx_base, const int32_t* __restrict__ idx_map) {
  const int i = blockIdx.x;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float acc = 0.f;
    for (int c = 0; c < n_chunks; ++c) acc += o_part[((int64_t)c * n_rows + i) * D + d];
    osum[(int64_t)i * D + d] = acc;
  }
  if (threadIdx.x == 0) {
    float acc = 0.f;
    for (int c = 0; c < n_chunks; ++c) acc += l_part[(int64_t)c * n_rows + i];
    lsum[i] = acc;
    if (topv) {
      float tv[KMAX];
      int32_t ti[KMAX];
      for (int q = 0; q < KMAX; ++q) {
        tv[q] = -INFINITY;
        ti[q] = -1;
      }
      if (is_out[i]) {
        for (int c = 0; c < n_chunks; ++c)
          for (int q = 0; q < k; ++q) {
            const float v = topv_part[((int64_t)c * n_rows + i) * k + q];
            if (v > tv[k - 1]) topk_insert<KMAX>(tv, ti, k, v, topi_part[((int64_t)c * n_rows + i) * k + q]);
          }
      }
      for (int q = 0; q < k; ++q) {
        topv[(int64_t)i * k + q] = tv[q];
        int32_t id = ti[q];
        if (id >= 0) id = (int32_t)(idx_base + (idx_map ? idx_map[id] : id));   // -> global slot
        topi[(int64_t)i * k + q] = id;
      }
    }
  }
}

// The same reduction for up to three sweeps in one launch (blockIdx.y = sweep): the merged main + side launch of the bf16 path.
struct ReduceJob {
  const float* l_part;
  const float* o_part;
  const float* topv_part;
  const int32_t* topi_part;
  int n_chunks;
  float* lsum;
  float* osum;
  float* topv;
  int32_t* topi;
  int64_t idx_base;
  const int32_t* idx_map;
};
struct ReduceJobs {
  ReduceJob j[3];
};
__global__ void __launch_bounds__(128) head_reduce_multi_kernel(const ReduceJobs jobs, int n_rows, int D, int k, const uint8_t* __restrict__ is_out) {
  const ReduceJob& r = jobs.j[blockIdx.y];
  const int i = blockIdx.x;
  const int n_chunks = r.n_chunks;
  const bool no_o = is_out[i] != 0;      // a hard-negative-only row has no softmax term: its O partials may not even have been written
  for (int d = threadIdx.x * 4; d < D; d += blockDim.x * 4) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c = 0; c < n_chunks && !no_o; ++c) {
      const float4 v = *reinterpret_cast<const float4*>(r.o_part + ((int64_t)c * n_rows + i) * D + d);
      acc.x += v.x;
      acc.y += v.y;
      acc.z += v.z;
      acc.w += v.w;
    }
    *reinterpret_cast<float4*>(r.osum + (int64_t)i * D + d) = acc;
  }
  if (threadIdx.x == 96) {      // scalar part (denominator, top-k merge) on one lane of the last warp
    float acc = 0.f;
    for (int c = 0; c < n_chunks; ++c) acc += r.l_part[(int64_t)c * n_rows + i];
    r.lsum[i] = acc;
    float tv[KMAX];
    int32_t ti[KMAX];
    for (int q = 0; q < KMAX; ++q) {
      tv[q] = -INFINITY;
      ti[q] = -1;
    }
    if (is_out[i]) {
      for (int c = 0; c < n_chunks; ++c)
        for (int q = 0; q < k; ++q) {
          const float v = r.topv_part[((int64_t)c * n_rows + i) * k + q];
          if (v > tv[k - 1]) topk_insert<KMAX>(tv, ti, k, v, r.topi_part[((int64_t)c * n_rows + i) * k + q]);
        }
    }
    for (int q = 0; q < k; ++q) {
      r.topv[(int64_t)i * k + q] = tv[q];
      int32_t id = ti[q];
      if (id >= 0) id = (int32_t)(r.idx_base + (r.idx_map ? r.idx_map[id] : id));   // -> global slot
      r.topi[(int64_t)i * k + q] = id;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// finalize
// ------------------------------------------------------------------------------------------------
struct FinalizeArgs {
  const float* P;              // [n][D]  (fp32 embeddings; only for nothing but kept for symmetry)
  const float* qf;             // [2][q_local][D]
  const __nv_bfloat16* qh;
  int use_bf16_rows;           // gather W rows from the bf16 mirror (consistent with the tensor-core sweep)
  const int32_t* label;
  const int32_t* tcol;
  const int32_t* tpos;
  const uint8_t* is_out;
  const int32_t* counts;
  const float* lsum;           // [4][n]
  const float* osum;           // [4][n][D]
  const float* tgt;            // [4][n]
  const float* topv;           // [n_ranks][3][n][k]
  const int32_t* topi;
  int n_ranks;
  int n, D, k;
  int64_t q_local, col_offset;
  int loss_type;
  float scale, margin, fixed_max;
  double cos_m, sin_m;         // cos / sin of the margin (Arc), computed once on the host
  float* row_loss;
  float* dp;
  // Overlay (sharded head with ONE exchange point per step, ffc_b200/dist.py): a queue row that has been rewritten since this pass's
  // sweep -- restored after a rollback pass, or enqueued by the commit pass that followed -- is read from where its sweep-time
  // content still is.  ovl_map[row * q_local + slot] = -1, or the source row: bit 30 clear -> ovl_g + idx * D (the gathered gallery
  // embedding that sat there), bit 30 set -> ovl_undo + idx * D (the previous content a later enqueue saved).  fp32 rows, rounded to
  // bf16 on the fly exactly as the mirror was.
  const int32_t* ovl_map;
  const float* ovl_g;
  const float* ovl_undo;
  // Optional export of the per-row scalars (queue-gradient mode, ffc_head_dqueue): coef [4][n] (cO loss 1 / 2, cT loss 1 / 2), the
  // hard-negative slot lists of outlier rows
  float* coef_out;
  int32_t* nslot_out;
  int32_t* wslot_out;
  uint8_t* wrow_out;
  // Output routing (reduce-scatter folded into finalize): with dp_peer != NULL row i of this rank's partial dLoss/dp is stored to
  // dp_peer[i / dp_rows_per_rank] + dp_slot_off + (i % dp_rows_per_rank) * D -- the owner rank's peer-mapped staging buffer
  // (stores travel over NVLink) -- instead of dp[i * D].
  float* const* dp_peer;
  int dp_rows_per_rank;
  int64_t dp_slot_off;
};

__device__ __forceinline__ float w_elem(const FinalizeArgs& a, int r, int64_t local_slot, int d) {
  const int64_t off = ((int64_t)r * a.q_local + local_slot) * a.D + d;
  return a.use_bf16_rows ? __bfloat162float(a.qh[off]) : a.qf[off];
}

// The scalar part of finalize for one row: margin function, log/exp in fp64, top-k merge.  `lsum_at(slot)` returns the row's
// softmax denominator of stats slot 0..3, `top_at(r, set, q, v, idx)` the q-th top-k candidate of rank r / column set `set`.
// T = double: the check mode and the statistics-in-the-middle path (1e-5 parity); T = float: the fused bf16 path, whose tolerance is
// 1e-2 -- the ~100 dependent operations per row are then 1-2 us of latency instead of the 16 us the fp64 pipe takes.
template <class T, class LsumF, class TgtF, class TopF>
__device__ __forceinline__ void row_coef_math(const FinalizeArgs& a, int i, int n_ranks, LsumF lsum_at, TgtF tgt_at, TopF top_at, float& loss_out, float (&cO)[2],
                                              float (&cT)[2], int& nw_out, int32_t* wslot_out, uint8_t* wrow_out) {
  const int n = a.n, k = a.k;
  const int n_pos = a.counts[0], n_out = a.counts[1];
  const bool outl = a.is_out[i];
  float loss = 0.f;
  cO[0] = cO[1] = cT[0] = cT[1] = 0.f;
  int nw = 0;
  if (!outl) {
    const T s = (T)a.scale, M = (T)a.fixed_max, m = (T)a.margin, cm = (T)a.cos_m, sm = (T)a.sin_m, one = (T)1;
    for (int l = 0; l < 2; ++l) {
      T ct = (T)tgt_at(l);
      // bf16 operands are rounded, so a cosine of two (nearly) identical unit vectors can land a few ulp outside
      // [-1, 1] and turn ffc.py:101's sqrt into NaN where the fp32 reference is finite: keep it strictly inside.
      // The fp32 check mode does not clamp and propagates NaN exactly like the reference.
      if (a.use_bf16_rows) ct = fmin(fmax(ct, (T)(-1.0 + 1e-6)), (T)(1.0 - 1e-6));
      T ft, dft;
      if (a.loss_type == FFC_LOSS_AM) {
        ft = ct - m;
        dft = one;
      } else if (a.loss_type == FFC_LOSS_ARC) {
        const T sn = sqrt((one - ct) * (one + ct));      // = sqrt(1 - ct^2) without the cancellation; NaN for |ct| > 1, like ffc.py:101
        ft = ct * cm - sn * sm;
        dft = cm + ct * sm / sn;
      } else {
        ft = ct > m ? ct - m : ct;
        dft = one;
      }
      const T zt = s * ft;
      const T et = exp(zt - M);
      const int cs = a.loss_type == FFC_LOSS_SV ? l : 0;   // common-statistics slot
      const T L = (T)lsum_at(cs) + (T)lsum_at(2 + l) + et;
      loss += (float)((log(L) + M - zt) / (T)n_pos);
      cO[l] = (float)(s / L / (T)n_pos);
      cT[l] = (float)(s * (et / L - one) * dft / (T)n_pos);
    }
  } else {
    // merge top-k candidates per loss: common (all ranks) + side_l (all ranks)
    const float wneg = 1.f / ((float)n_out * (float)k);
    cO[0] = wneg;
    for (int l = 0; l < 2; ++l) {
      float tv[KMAX];
      int32_t ti[KMAX];
      for (int q = 0; q < KMAX; ++q) {
        tv[q] = -INFINITY;
        ti[q] = -1;
      }
      for (int r = 0; r < n_ranks; ++r)
        for (int src = 0; src < 2; ++src) {
          const int set = src == 0 ? 0 : 1 + l;
          for (int q = 0; q < k; ++q) {
            float v;
            int32_t idx;
            top_at(r, set, q, v, idx);
            // a side entry is tagged in bit 30: under loss 2 it reads queue[1]
            if (!(v > tv[k - 1])) break;      // every candidate list is sorted: nothing further of this one can enter
            topk_insert<KMAX>(tv, ti, k, v, (int32_t)(idx | (src ? 0x40000000 : 0)));
          }
        }
      for (int q = 0; q < k; ++q) {
        if (ti[q] < 0) continue;
        const float v = tv[q];
        loss += (v > 0.f ? v : 0.f) * wneg;
        if (v >= 0.f) {
          wslot_out[nw] = ti[q] & 0x3fffffff;
          wrow_out[nw] = (ti[q] & 0x40000000) ? (uint8_t)l : (uint8_t)0;
          ++nw;
        }
      }
    }
  }
  loss_out = loss;
  nw_out = nw;
}

// Pass 1, one THREAD per row: the scalar part of finalize.  Doing this per thread instead of on thread 0 of a per-row block
// keeps the fp64 transcendental latency off the critical path.
__global__ void __launch_bounds__(128) head_row_coef_kernel(const FinalizeArgs a, float* __restrict__ coef, int32_t* __restrict__ nslot,
                                                            int32_t* __restrict__ wslot, uint8_t* __restrict__ wrow) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = a.n, k = a.k;
  if (i >= n) return;
  float loss, cO[2], cT[2];
  int nw;
  row_coef_math<double>(
      a, i, a.n_ranks, [&](int slot) { return a.lsum[slot * n + i]; }, [&](int l) { return a.tgt[l * n + i]; },
      [&](int r, int set, int q, float& v, int32_t& idx) {
        const int64_t base = ((((int64_t)r * 3 + set) * n) + i) * k;
        v = a.topv[base + q];
        idx = a.topi[base + q];
      },
      loss, cO, cT, nw, wslot + (int64_t)i * 2 * KMAX, wrow + (int64_t)i * 2 * KMAX);
  a.row_loss[i] = loss;
  coef[0 * n + i] = cO[0];
  coef[1 * n + i] = cO[1];
  coef[2 * n + i] = cT[0];
  coef[3 * n + i] = cT[1];
  nslot[i] = nw;
}

// Per-rank record exchanged by the sharded head (4-byte words, n = rows, k = top-k):
//   [0, 8n)          float  red[8][n]     lsum slots 0..3 (common loss 1, unused, side 0, side 1), tgt slots 0..3
//   [8n, 8n+3nk)     float  topv[3][n][k]
//   [8n+3nk, +3nk)   int32  topi[3][n][k] GLOBAL slots
__host__ __device__ __forceinline__ int64_t record_words(int64_t n, int64_t k) { return 8 * n + 6 * n * k; }

// Chunk reduction of the three sweeps' SCALAR partials (softmax denominators, top-k candidates) straight into this rank's
// record; the O partials stay where they are for head_finalize_fused_kernel<true>.  One thread per (row, sweep).
__global__ void __launch_bounds__(128) head_reduce_scalars_kernel(const ReduceJobs jobs, int n, int k, const uint8_t* __restrict__ is_out,
                                                                  float* __restrict__ rec) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 3 * n) return;
  const int i = t / 3, w = t - 3 * i;
  const ReduceJob& r = jobs.j[w];
  float acc = 0.f;
  for (int c = 0; c < r.n_chunks; ++c) acc += r.l_part[(int64_t)c * n + i];
  rec[(int64_t)(w == 0 ? 0 : 1 + w) * n + i] = acc;
  if (w == 0) rec[(int64_t)1 * n + i] = 0.f;
  float tv[KMAX];
  int32_t ti[KMAX];
  for (int q = 0; q < KMAX; ++q) {
    tv[q] = -INFINITY;
    ti[q] = -1;
  }
  if (is_out[i]) {
    for (int c = 0; c < r.n_chunks; ++c)
      for (int q = 0; q < k; ++q) {
        const float v = r.topv_part[((int64_t)c * n + i) * k + q];
        if (v > tv[k - 1]) topk_insert<KMAX>(tv, ti, k, v, r.topi_part[((int64_t)c * n + i) * k + q]);
      }
  }
  float* topv = rec + 8 * (int64_t)n;
  int32_t* topi = reinterpret_cast<int32_t*>(rec + 8 * (int64_t)n + 3 * (int64_t)n * k);
  for (int q = 0; q < k; ++q) {
    int32_t id = ti[q];
    if (id >= 0) id = (int32_t)(r.idx_base + (r.idx_map ? r.idx_map[id] : id));   // -> global slot
    topv[((int64_t)w * n + i) * k + q] = tv[q];
    topi[((int64_t)w * n + i) * k + q] = id;
  }
}

// One prototype row as the fused finalize reads it: the bf16 mirror row, or (overlay) an fp32 row rounded on the fly.
struct WRow {
  const __nv_bfloat16* h;
  const float* f;
};
__device__ __forceinline__ WRow w_row(const FinalizeArgs& a, int r, int64_t loc) {
  WRow w;
  const int64_t e = (int64_t)r * a.q_local + loc;
  w.h = a.qh + e * a.D;
  w.f = nullptr;
  if (a.ovl_map) {
    const int32_t c = __ldg(a.ovl_map + e);
    if (c >= 0) w.f = (c & 0x40000000) ? a.ovl_undo + (int64_t)(c & 0x3fffffff) * a.D : a.ovl_g + (int64_t)c * a.D;
  }
  return w;
}
__device__ __forceinline__ float4 w_load4(const WRow& w, int d) {
  if (w.f) {
    const float4 v = *reinterpret_cast<const float4*>(w.f + d);
    return make_float4(__bfloat162float(__float2bfloat16(v.x)), __bfloat162float(__float2bfloat16(v.y)), __bfloat162float(__float2bfloat16(v.z)),
                       __bfloat162float(__float2bfloat16(v.w)));
  }
  const uint2 u = *reinterpret_cast<const uint2*>(w.h + d);
  const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162*>(&u.x), hi = *reinterpret_cast<const __nv_bfloat162*>(&u.y);
  const float2 a2 = __bfloat1622float2(lo), b2 = __bfloat1622float2(hi);
  return make_float4(a2.x, a2.y, b2.x, b2.y);
}

// Fast path of the bf16 AM / Arc head: chunk reduction of the three sweeps' partials, the scalar part and dLoss/dp in ONE
// launch.  No osum round trip through HBM; replaces reduce + row_coef + finalize.  A block takes FR = 4 rows (2 048 blocks at the 8-GPU
// row count: the partial sums are ~100 MB to read, and it takes that many loads in flight to read them at the HBM rate):
//   phase 1 (GATHERED = false only): one thread per (row, sweep) sums the chunk denominators and merges the chunk top-k lists;
//   phase 2: one THREAD per row does the scalar part (margin function, log / exp, top-k merge over ranks) -- in fp32, all rows of
//            the grid side by side (one lane per row on the fp64 pipe cost 16 us per row, 3.5 waves of it at 8 192 rows);
//   phase 3: one warp per row, lanes over D: chunk sums of the three O partials, the two prototype rows of the target (or the
//            hard-negative rows of an outlier row), 16-byte stores -- the bandwidth part, ~(chunks * 3 + 2) * D * 4 bytes per row.
//   GATHERED = false (one GPU): the scalars are reduced here from the partials as well;
//   GATHERED = true (sharded head): the scalars come from the n_ranks gathered records (`rec`, `rec_stride` words apart),
//     summed in rank order on every rank; O is this rank's partial, so dp is this rank's contribution -- stored locally for a
//     reduce-scatter, or (dp_peer) straight into the owner rank's staging buffer.
constexpr int FR = 4;
template <bool GATHERED>
__global__ void __launch_bounds__(128) head_finalize_fused_kernel(const ReduceJobs jobs, const FinalizeArgs a, const float* __restrict__ rec,
                                                                  int64_t rec_stride) {
  const int tid = threadIdx.x;
  const int row0 = blockIdx.x * FR, n = a.n, D = a.D, k = a.k;
  __shared__ float s_l[FR][3];
  __shared__ float s_tv[FR][3][KMAX];
  __shared__ int32_t s_ti[FR][3][KMAX];
  __shared__ float s_coef[FR][4];
  __shared__ int s_nw[FR];
  __shared__ int32_t s_wslot[FR][2 * KMAX];
  __shared__ uint8_t s_wrow[FR][2 * KMAX];
  __shared__ WRow s_t0[FR], s_t1[FR];
  if (!GATHERED) {
    if (tid < FR * 3) {
      const int r = tid / 3, j = tid - 3 * r, i = row0 + r;
      if (i < n) {
        const ReduceJob& rj = jobs.j[j];
        float acc = 0.f;
        for (int c = 0; c < rj.n_chunks; ++c) acc += rj.l_part[(int64_t)c * n + i];
        s_l[r][j] = acc;
        float tv[KMAX];
        int32_t ti[KMAX];
        for (int q = 0; q < KMAX; ++q) {
          tv[q] = -INFINITY;
          ti[q] = -1;
        }
        if (a.is_out[i]) {
          for (int c = 0; c < rj.n_chunks; ++c)
            for (int q = 0; q < k; ++q) {
              const float v = rj.topv_part[((int64_t)c * n + i) * k + q];
              if (v > tv[k - 1]) topk_insert<KMAX>(tv, ti, k, v, rj.topi_part[((int64_t)c * n + i) * k + q]);
            }
        }
        for (int q = 0; q < KMAX; ++q) {
          int32_t id = ti[q];
          if (id >= 0) id = (int32_t)(rj.idx_base + (rj.idx_map ? rj.idx_map[id] : id));   // -> global slot
          s_tv[r][j][q] = tv[q];
          s_ti[r][j][q] = id;
        }
      }
    }
    __syncthreads();
  }
  // GATHERED: the ranks' records are staged through shared memory by all threads -- per row 6 scalars x R ranks and, for an outlier
  // row, 3 candidate sets x R ranks x k (value, slot) pairs.  Read by the one thread that does the row's scalar part they were
  // ~50 (positive row) / ~500 (outlier row) dependent global loads: the latency of this phase paced the kernel at 8 ranks.
  constexpr int RS = 16;                       // ranks the staging is sized for (more: the records are read in place)
  __shared__ float s_red[GATHERED ? FR : 1][6][GATHERED ? RS : 1];
  __shared__ float s_cv[GATHERED ? FR : 1][3][GATHERED ? RS : 1][KMAX];
  __shared__ int32_t s_ci[GATHERED ? FR : 1][3][GATHERED ? RS : 1][KMAX];
  const bool staged = GATHERED && a.n_ranks <= RS;
  if (staged) {
    const int R = a.n_ranks;
    for (int e = tid; e < FR * 6 * R; e += 128) {
      const int r = e / (6 * R), j = (e / R) % 6, q = e % R, i = row0 + r;
      if (i < n) s_red[r][j][q] = rec[q * rec_stride + (int64_t)j * n + i];
    }
    for (int e = tid; e < FR * 3 * R * k; e += 128) {
      const int r = e / (3 * R * k), set = (e / (R * k)) % 3, q = (e / k) % R, x = e % k, i = row0 + r;
      if (i < n && a.is_out[i]) {
        const float* base = rec + q * rec_stride + 8 * (int64_t)n;
        const int64_t o = ((int64_t)set * n + i) * k + x;
        s_cv[r][set][q][x] = base[o];
        s_ci[r][set][q][x] = reinterpret_cast<const int32_t*>(base + 3 * (int64_t)n * k)[o];
      }
    }
    __syncthreads();
  }
  if (tid < FR && row0 + tid < n) {
    const int r = tid, i = row0 + r;
    float loss, cO[2], cT[2];
    int nw;
    if (staged) {
      const int R = a.n_ranks;
      row_coef_math<float>(
          a, i, R,
          [&](int slot) {
            float acc = 0.f;
            for (int q = 0; q < R; ++q) acc += s_red[r][slot][q];      // rank order: the same sum on every rank
            return acc;
          },
          [&](int l) {
            float acc = 0.f;
            for (int q = 0; q < R; ++q) acc += s_red[r][4 + l][q];
            return acc;
          },
          [&](int q, int set, int e, float& v, int32_t& idx) {
            v = s_cv[r][set][q][e];
            idx = s_ci[r][set][q][e];
          },
          loss, cO, cT, nw, s_wslot[r], s_wrow[r]);
    } else if (GATHERED) {
      const int R = a.n_ranks;
      row_coef_math<float>(
          a, i, R,
          [&](int slot) {
            float acc = 0.f;
            for (int q = 0; q < R; ++q) acc += rec[q * rec_stride + (int64_t)slot * n + i];
            return acc;
          },
          [&](int l) {
            float acc = 0.f;
            for (int q = 0; q < R; ++q) acc += rec[q * rec_stride + (int64_t)(4 + l) * n + i];
            return acc;
          },
          [&](int q, int set, int e, float& v, int32_t& idx) {
            const float* base = rec + q * rec_stride + 8 * (int64_t)n;
            const int64_t o = ((int64_t)set * n + i) * k + e;
            v = base[o];
            idx = reinterpret_cast<const int32_t*>(base + 3 * (int64_t)n * k)[o];
          },
          loss, cO, cT, nw, s_wslot[r], s_wrow[r]);
    } else {
      row_coef_math<float>(
          a, i, 1, [&](int slot) { return slot == 0 ? s_l[r][0] : (slot >= 2 ? s_l[r][slot - 1] : 0.f); }, [&](int l) { return a.tgt[l * n + i]; },
          [&](int, int set, int e, float& v, int32_t& idx) {
            v = s_tv[r][set][e];
            idx = s_ti[r][set][e];
          },
          loss, cO, cT, nw, s_wslot[r], s_wrow[r]);
    }
    a.row_loss[i] = loss;
    s_coef[r][0] = cO[0];
    s_coef[r][1] = cO[1];
    s_coef[r][2] = cT[0];
    s_coef[r][3] = cT[1];
    s_nw[r] = nw;
    if (a.coef_out) {
      a.coef_out[0 * n + i] = cO[0];
      a.coef_out[1 * n + i] = cO[1];
      a.coef_out[2 * n + i] = cT[0];
      a.coef_out[3 * n + i] = cT[1];
      a.nslot_out[i] = nw;
      for (int x = 0; x < nw; ++x) {
        a.wslot_out[(int64_t)i * 2 * KMAX + x] = s_wslot[r][x];
        a.wrow_out[(int64_t)i * 2 * KMAX + x] = s_wrow[r][x];
      }
    }
  }
  if (tid < FR && row0 + tid < n) {      // the rows' prototype rows (through the overlay), resolved once per row
    const int i = row0 + tid;
    const int32_t tc = a.tcol[i];
    WRow t0, t1;
    t0.h = t1.h = nullptr;
    t0.f = t1.f = nullptr;
    if (!a.is_out[i] && tc >= 0) {
      t0 = w_row(a, 0, tc);
      t1 = w_row(a, (a.tpos[i] >= 0) ? 1 : 0, tc);
    }
    s_t0[tid] = t0;
    s_t1[tid] = t1;
  }
  __syncthreads();
  // phase 3: (row, 4 features) items dealt to the 128 threads; the chunk loads of an item are independent (issued eight at a time,
  // added in chunk order) -- with one warp per row and a serial chunk loop the kernel ran at memory LATENCY (70 us for 2 048 rows x
  // 9 chunks: 37 MB)
  const int D4 = D >> 2;
  const int64_t cstride = (int64_t)n * D;
  for (int item = tid; item < FR * D4; item += 128) {
    const int r = item / D4, d = (item - r * D4) * 4;
    const int i = row0 + r;
    if (i >= n) break;
    const bool outl = a.is_out[i];
    float* out = a.dp_peer ? a.dp_peer[i / a.dp_rows_per_rank] + a.dp_slot_off + (int64_t)(i % a.dp_rows_per_rank) * D : a.dp + (int64_t)i * D;
    float g[4] = {0.f, 0.f, 0.f, 0.f};
    if (!outl) {
      const float cO0 = s_coef[r][0], cO1 = s_coef[r][1], cT0 = s_coef[r][2], cT1 = s_coef[r][3];
      float o[3][4];
#pragma unroll
      for (int jb = 0; jb < 3; ++jb) {
        const ReduceJob& rj = jobs.j[jb];
        const float* base = rj.o_part + (int64_t)i * D + d;
        const int nc = rj.n_chunks;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int c = 0;
        for (; c + 8 <= nc; c += 8) {
          float4 v[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) v[u] = __ldcs(reinterpret_cast<const float4*>(base + (c + u) * cstride));
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            acc.x += v[u].x;
            acc.y += v[u].y;
            acc.z += v[u].z;
            acc.w += v[u].w;
          }
        }
        for (; c + 2 <= nc; c += 2) {
          const float4 v0 = __ldcs(reinterpret_cast<const float4*>(base + c * cstride));
          const float4 v1 = __ldcs(reinterpret_cast<const float4*>(base + (c + 1) * cstride));
          acc.x += v0.x;
          acc.y += v0.y;
          acc.z += v0.z;
          acc.w += v0.w;
          acc.x += v1.x;
          acc.y += v1.y;
          acc.z += v1.z;
          acc.w += v1.w;
        }
        for (; c < nc; ++c) {
          const float4 v = __ldcs(reinterpret_cast<const float4*>(base + c * cstride));
          acc.x += v.x;
          acc.y += v.y;
          acc.z += v.z;
          acc.w += v.w;
        }
        o[jb][0] = acc.x;
        o[jb][1] = acc.y;
        o[jb][2] = acc.z;
        o[jb][3] = acc.w;
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) g[e] = cO0 * (o[0][e] + o[1][e]) + cO1 * (o[0][e] + o[2][e]);
      const WRow t0 = s_t0[r], t1 = s_t1[r];
      if (t0.h) {
        const float4 w0 = w_load4(t0, d), w1 = w_load4(t1, d);
        g[0] += cT0 * w0.x + cT1 * w1.x;
        g[1] += cT0 * w0.y + cT1 * w1.y;
        g[2] += cT0 * w0.z + cT1 * w1.z;
        g[3] += cT0 * w0.w + cT1 * w1.w;
      }
    } else {
      const float cO0 = s_coef[r][0];
      const int nw = s_nw[r];
      for (int x = 0; x < nw; ++x) {
        const int64_t loc = (int64_t)s_wslot[r][x] - a.col_offset;
        if (loc >= 0 && loc < a.q_local) {
          const float4 wv = w_load4(w_row(a, s_wrow[r][x], loc), d);
          g[0] += cO0 * wv.x;
          g[1] += cO0 * wv.y;
          g[2] += cO0 * wv.z;
          g[3] += cO0 * wv.w;
        }
      }
    }
    *reinterpret_cast<float4*>(out + d) = make_float4(g[0], g[1], g[2], g[3]);
  }
  // rows stored into a peer's staging buffer: make them visible system-wide before this kernel counts as finished -- the flag that
  // tells the peer "my rows are there" is written by the next launch in the stream (ffc_sum_slabs_barrier)
  if (a.dp_peer) __threadfence_system();
}

// Pass 2, one block per row: dLoss/dp from the accumulated sums (bandwidth bound).
__global__ void __launch_bounds__(128) head_finalize_kernel(const FinalizeArgs a, const float* __restrict__ coef, const int32_t* __restrict__ nslot,
                                                            const int32_t* __restrict__ wslot, const uint8_t* __restrict__ wrow) {
  const int i = blockIdx.x, n = a.n, D = a.D;
  const bool outl = a.is_out[i];
  const float cO0 = coef[0 * n + i], cO1 = coef[1 * n + i], cT0 = coef[2 * n + i], cT1 = coef[3 * n + i];
  const int32_t tc = a.tcol[i];
  const int trow2 = (a.tpos[i] >= 0) ? 1 : 0;
  const int nw = nslot[i];
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float g = 0.f;
    if (!outl) {
      const float oc0 = a.osum[((int64_t)0 * n + i) * D + d];
      const float oc1 = a.loss_type == FFC_LOSS_SV ? a.osum[((int64_t)1 * n + i) * D + d] : oc0;
      g = cO0 * (oc0 + a.osum[((int64_t)2 * n + i) * D + d]) + cO1 * (oc1 + a.osum[((int64_t)3 * n + i) * D + d]);
      if (tc >= 0) g += cT0 * w_elem(a, 0, tc, d) + cT1 * w_elem(a, trow2, tc, d);
    } else {
      for (int e = 0; e < nw; ++e) {
        const int64_t loc = (int64_t)wslot[(int64_t)i * 2 * KMAX + e] - a.col_offset;
        if (loc >= 0 && loc < a.q_local) g += cO0 * w_elem(a, wrow[(int64_t)i * 2 * KMAX + e], loc, d);
      }
    }
    a.dp[(int64_t)i * D + d] = g;
  }
}

__global__ void __launch_bounds__(1024) head_loss_sum_kernel(const float* __restrict__ row_loss, int n, float* loss_out) {
  __shared__ double sh[1024];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += 1024) acc += row_loss[i];
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) loss_out[0] = (float)sh[0];
}

__global__ void head_p_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = __float2bfloat16(src[i]);
}

// The softmax reference point M.  The logits are bounded by construction (unit-norm rows: |cos| <= 1), z in [z_min, z_max] with
// z_max = scale (SV: scale * (2t - 1), ffc.py:124), z_min = -scale, so a FIXED reference is exact as long as every e^(z - M) and
// their sum over the queue stay normal fp32 numbers: M >= z_max - 67 (2^30 columns of e^67 < 2^127) and M <= z_min + 87.  M is the
// midpoint of that window, (z_max + z_min + 20) / 2 -- 10 for AM / Arc at ANY scale, e.g. the customary ArcFace s = 64: nothing is
// flushed, nothing overflows, no rescaling of the accumulators is ever needed.  (M = scale, the usual "subtract the largest
// possible logit", would push e^(z_min - M) = e^(-2 scale) below the normal range for scale >= 43.5.)
static float logit_max_of(const ffc_head_config& c) { return c.loss_type == FFC_LOSS_SV ? c.scale * (2.f * SV_T - 1.f) : c.scale; }
static float fixed_max_of(const ffc_head_config& c) { return 0.5f * (logit_max_of(c) - c.scale + 20.f); }
static bool fixed_max_ok(const ffc_head_config& c) { return c.scale > 0.f && logit_max_of(c) + c.scale <= 154.f; }

}  // namespace ffc

using namespace ffc;

extern "C" int ffc_head_stats_bytes(const ffc_head_config* cfg, int n_rows, int64_t sizes_out[5]) {
  FFC_REQUIRE(cfg && sizes_out && n_rows >= 0, "ffc_head_stats_bytes: bad arguments");
  const int64_t n = n_rows, D = cfg->feat_dim, k = cfg->topk;
  sizes_out[0] = 4 * n * sizeof(float);
  sizes_out[1] = 4 * n * D * sizeof(float);
  sizes_out[2] = 4 * n * sizeof(float);
  sizes_out[3] = 3 * n * k * sizeof(float);
  sizes_out[4] = 3 * n * k * sizeof(int32_t);
  return FFC_OK;
}

extern "C" int ffc_head_create(const ffc_head_config* cfg, ffc_head_t** out) {
  FFC_REQUIRE(cfg && out, "ffc_head_create: NULL argument");
  FFC_REQUIRE(cfg->max_rows >= 1 && cfg->q_local >= 1 && cfg->q_total >= cfg->q_local && cfg->col_offset >= 0, "ffc_head_create: bad sizes");
  FFC_REQUIRE(cfg->q_total < 0x40000000, "ffc_head_create: queue size must be below 2^30");
  FFC_REQUIRE(cfg->feat_dim >= 4 && cfg->feat_dim % 4 == 0 && cfg->feat_dim <= 512, "ffc_head_create: feat_dim %d (multiple of 4, <= 512)", cfg->feat_dim);
  FFC_REQUIRE(cfg->loss_type >= 0 && cfg->loss_type <= 2, "ffc_head_create: loss_type %d", cfg->loss_type);
  FFC_REQUIRE(cfg->topk >= 1 && cfg->topk <= KMAX, "ffc_head_create: topk %d outside [1,%d]", cfg->topk, KMAX);
  FFC_REQUIRE(cfg->precision == FFC_PREC_BF16 || cfg->precision == FFC_PREC_FP32, "ffc_head_create: precision %d", cfg->precision);
  if (cfg->precision == FFC_PREC_BF16) {
    FFC_REQUIRE(cfg->feat_dim == 64 || cfg->feat_dim == 128 || cfg->feat_dim == 256 || cfg->feat_dim == 512,
                "ffc_head_create: the bf16 tensor-core path is built for feat_dim 64, 128, 256 or 512 (got %d); other widths: FFC_PREC_FP32",
                cfg->feat_dim);
  }
  FFC_REQUIRE(fixed_max_ok(*cfg), "ffc_head_create: scale %.1f outside (0, %.1f]: the logit range must fit the fp32 exponent range around the fixed softmax reference",
              cfg->scale, cfg->loss_type == FFC_LOSS_SV ? 154.f / (2.f * SV_T) : 77.f);
  ffc_head* h = new ffc_head();
  memset(h, 0, sizeof(*h));
  h->cfg = *cfg;
  const int64_t R = cfg->max_rows, D = cfg->feat_dim;
  h->part_rows_cap = std::max<int64_t>(20 * R, 40960);
  h->max_chunks = 1024;
  FFC_CUDA(cudaMalloc(&h->p16, R * D * sizeof(__nv_bfloat16)));
  FFC_CUDA(cudaMalloc(&h->side_f32, 2 * R * D * sizeof(float)));
  FFC_CUDA(cudaMalloc(&h->side_bf16, 2 * R * D * sizeof(__nv_bfloat16)));
  FFC_CUDA(cudaMalloc(&h->tcol, R * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->tpos, R * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->is_out, R));
  FFC_CUDA(cudaMalloc(&h->kth_shared, R * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->thr, 2 * R * sizeof(float)));
  FFC_CUDA(cudaMalloc(&h->counts, 4 * sizeof(int32_t)));
  FFC_CUDA(cudaMemset(h->counts, 0, 4 * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->row_map, R * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->part_ctr, 2 * sizeof(int32_t)));
  FFC_CUDA(cudaMemset(h->part_ctr, 0, 2 * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->row_loss, R * sizeof(float)));
  FFC_CUDA(cudaMalloc(&h->coef, 4 * R * sizeof(float)));
  FFC_CUDA(cudaMalloc(&h->nslot, R * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->wslot, R * 2 * KMAX * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->wrow, R * 2 * KMAX));
  FFC_CUDA(cudaMalloc(&h->l_part, h->part_rows_cap * sizeof(float)));
  FFC_CUDA(cudaMalloc(&h->o_part, h->part_rows_cap * D * sizeof(float)));
  FFC_CUDA(cudaMalloc(&h->topv_part, h->part_rows_cap * KMAX * sizeof(float)));
  FFC_CUDA(cudaMalloc(&h->topi_part, h->part_rows_cap * KMAX * sizeof(int32_t)));
  if (cfg->precision == FFC_PREC_BF16) h->sm100 = sm100_cache_create();
  h->ev = new std::vector<cudaEvent_t>();
  h->jobs = new ReduceJobs();
  *out = h;
  return FFC_OK;
}

extern "C" int ffc_head_destroy(ffc_head_t* h) {
  if (!h) return FFC_OK;
  cudaFree(h->p16);
  cudaFree(h->side_f32);
  cudaFree(h->side_bf16);
  cudaFree(h->tcol);
  cudaFree(h->tpos);
  cudaFree(h->is_out);
  cudaFree(h->row_map);
  cudaFree(h->part_ctr);
  cudaFree(h->kth_shared);
  cudaFree(h->pc16);
  cudaFree(h->dq_col);
  cudaFree(h->dq_l);
  cudaFree(h->dq_tv);
  cudaFree(h->dq_ti);
  cudaFree(h->dq_claim);
  cudaFree(h->thr);
  cudaFree(h->counts);
  cudaFree(h->row_loss);
  cudaFree(h->coef);
  cudaFree(h->nslot);
  cudaFree(h->wslot);
  cudaFree(h->wrow);
  cudaFree(h->l_part);
  cudaFree(h->o_part);
  cudaFree(h->topv_part);
  cudaFree(h->topi_part);
  if (h->sm100) sm100_cache_destroy(h->sm100);
  if (h->ev) {
    for (cudaEvent_t e : *h->ev) cudaEventDestroy(e);
    delete h->ev;
  }
  delete h->jobs;
  delete h;
  return FFC_OK;
}

static int run_one_sweep(ffc_head* h, SweepArgs a, int cache_slot, int stat_slot, int top_slot, const ffc_head_stats* out, int64_t idx_base,
                         const int32_t* idx_map, cudaStream_t s) {
  const bool bf16 = h->cfg.precision == FFC_PREC_BF16;
  a.n_chunks = bf16 ? sm100_pick_chunks(a.n_rows, a.n_cols, a.D, (int)std::min<int64_t>(h->part_rows_cap / std::max(1, a.n_rows), h->max_chunks)) : simt_pick_chunks(a.n_rows, a.n_cols);
  FFC_REQUIRE((int64_t)a.n_chunks * a.n_rows <= h->part_rows_cap && a.n_chunks <= h->max_chunks, "head sweep: partial workspace too small (%d chunks x %d rows)",
              a.n_chunks, a.n_rows);
  a.l_part = h->l_part;
  a.o_part = h->o_part;
  a.topv_part = h->topv_part;
  a.topi_part = h->topi_part;
  const bool timed = h->timing && cache_slot == 0;
  if (timed) {
    if (h->ev_used + 2 > h->ev->size()) {
      for (int e = 0; e < 2; ++e) {
        cudaEvent_t ev;
        FFC_CUDA(cudaEventCreate(&ev));
        h->ev->push_back(ev);
      }
    }
    FFC_CUDA(cudaEventRecord((*h->ev)[h->ev_used], s));
  }
  int rc = bf16 ? launch_sweep_sm100(h->sm100, cache_slot, a, s) : launch_sweep_simt(a, s);
  if (rc) return rc;
  if (timed) {
    FFC_CUDA(cudaEventRecord((*h->ev)[h->ev_used + 1], s));
    h->ev_used += 2;
  }
  const int n = a.n_rows, D = a.D, k = a.k;
  head_reduce_kernel<<<n, 128, 0, s>>>(a.l_part, a.o_part, a.topv_part, a.topi_part, a.n_chunks, n, D, k, out->lsum + (int64_t)stat_slot * n,
                                       out->osum + (int64_t)stat_slot * n * D, top_slot >= 0 ? out->topv + (int64_t)top_slot * n * k : nullptr,
                                       top_slot >= 0 ? out->topi + (int64_t)top_slot * n * k : nullptr, a.is_out, idx_base, idx_map);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

// bf16, AM / Arc: the main sweep over queue[0] and the two side sweeps over the gathered `ones` rows of queue[0] / queue[1] as ONE
// launch of the tcgen05 kernel (their items are concatenated), followed by one reduce launch.
static int run_merged_sweeps(ffc_head* h, SweepArgs a, const ffc_head_pass* in, const ffc_head_stats* out, bool defer_reduce, cudaStream_t s) {
  const ffc_head_config& c = h->cfg;
  const int n = a.n_rows, D = a.D, k = a.k;
  SweepArgs sw[3];
  ReduceJobs jobs;
  int64_t part_row = 0;
  for (int i = 0; i < 3; ++i) {
    SweepArgs& w = sw[i];
    w = a;
    if (i == 0) {
      w.W_bf16 = (const __nv_bfloat16*)in->queue_bf16;
      w.n_cols = c.q_local;
      w.n_cols_dev = nullptr;
      w.tcol = h->tcol;
      w.cmask = in->cmask;
      w.n_chunks = sm100_pick_chunks(n, w.n_cols, D, (int)std::min<int64_t>(h->part_rows_cap / std::max(1, n) - 2, h->max_chunks));   // - the two side sweeps' partials
    } else {
      w.W_bf16 = h->side_bf16 + (int64_t)(i - 1) * c.max_rows * D;
      w.n_cols = c.max_rows;
      w.n_cols_dev = in->n_ones;
      w.tcol = h->tpos;
      w.cmask = nullptr;
      w.n_chunks = 1;
    }
    w.thr = nullptr;
    w.l_part = h->l_part + part_row;
    w.o_part = h->o_part + part_row * D;
    w.topv_part = h->topv_part + part_row * k;
    w.topi_part = h->topi_part + part_row * k;
    const int stat_slot = i == 0 ? 0 : 1 + i, top_slot = i;
    ReduceJob& r = jobs.j[i];
    r.l_part = w.l_part;
    r.o_part = w.o_part;
    r.topv_part = w.topv_part;
    r.topi_part = w.topi_part;
    r.n_chunks = w.n_chunks;
    r.lsum = out->lsum + (int64_t)stat_slot * n;
    r.osum = out->osum + (int64_t)stat_slot * n * D;
    r.topv = out->topv + (int64_t)top_slot * n * k;
    r.topi = out->topi + (int64_t)top_slot * n * k;
    r.idx_base = c.col_offset;
    r.idx_map = i == 0 ? nullptr : in->ones_list;
    part_row += (int64_t)w.n_chunks * n;
  }
  FFC_REQUIRE(part_row <= h->part_rows_cap && sw[0].n_chunks <= h->max_chunks, "head sweep: partial workspace too small (%d chunks x %d rows)",
              sw[0].n_chunks, n);
  const bool timed = h->timing != 0;
  if (timed) {
    if (h->ev_used + 2 > h->ev->size()) {
      for (int e = 0; e < 2; ++e) {
        cudaEvent_t ev;
        FFC_CUDA(cudaEventCreate(&ev));
        h->ev->push_back(ev);
      }
    }
    FFC_CUDA(cudaEventRecord((*h->ev)[h->ev_used], s));
  }
  int rc = launch_sweeps_sm100(h->sm100, sw, 3, s);
  if (rc) return rc;
  if (timed) {
    FFC_CUDA(cudaEventRecord((*h->ev)[h->ev_used + 1], s));
    h->ev_used += 2;
  }
  *h->jobs = jobs;
  h->jobs_pending = defer_reduce ? 1 : 0;
  if (!defer_reduce) {
    head_reduce_multi_kernel<<<dim3(n, 3), 128, 0, s>>>(jobs, n, D, k, a.is_out);
    FFC_LAUNCH_CHECK();
  }
  return FFC_OK;
}

// SV on a sharded queue: the hard-example threshold (ffc.py:122, gt - margin) of a row whose target column lives on another rank.
// tgt holds the all-reduced target cosines ([0], [1]) and owner count ([2]) written by the ranks' prep launches.
__global__ void __launch_bounds__(128) head_thr_from_tgt_kernel(const float* __restrict__ tgt, int n, float margin, float* __restrict__ thr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const bool has = tgt[2 * n + i] > 0.f;
  thr[i] = has ? tgt[i] - margin : INFINITY;
  thr[n + i] = has ? tgt[n + i] - margin : INFINITY;
}

// The merged bf16 AM / Arc sweep takes its rows in "hard-negative-only rows last" order when the launch is several waves of work items
// deep (the 4- / 8-way shard shapes): row tiles made of such rows then cost about half a tile (no exponentials, no GEMM-2) and the
// hardware deals the items out as pairs free up.  In a one-wave launch (C2, C4 on one GPU) the kernel ends with its slowest item, and
// concentrating the hard-negative scans in a few items makes that one slower (C2: +11 %), so the identity order stays.
// FFC_SWEEP_NO_ROWMAP=1: never (A/B measurements); FFC_SWEEP_ROWMAP=1: at any shape (tests).  SV sweeps and the check mode do not use it.
static bool use_row_map(const ffc_head* h, int n_rows) {
  static const bool off = getenv("FFC_SWEEP_NO_ROWMAP") != nullptr && atoi(getenv("FFC_SWEEP_NO_ROWMAP")) != 0;
  static const bool force = getenv("FFC_SWEEP_ROWMAP") != nullptr && atoi(getenv("FFC_SWEEP_ROWMAP")) != 0;      // tests: at any shape
  if (off || h->cfg.precision != FFC_PREC_BF16 || h->cfg.loss_type == FFC_LOSS_SV) return false;
  if (force) return true;
  const int row_tiles = (n_rows + 127) / 128;
  const int chunks = sm100_pick_chunks(n_rows, h->cfg.q_local, h->cfg.feat_dim, (int)std::min<int64_t>(h->part_rows_cap / std::max(1, n_rows) - 2, h->max_chunks));
  return (int64_t)row_tiles * chunks > 2 * 74;
}

// phase: 1 = prep only, 2 = sweeps only (prep was run by ffc_head_prep; SV thresholds are re-derived from out->tgt), 3 = both
static int head_sweep_impl(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* out, bool defer_reduce, void* stream, int phase = 3) {
  FFC_REQUIRE(h && in && out, "ffc_head_sweep: NULL argument");
  h->jobs_pending = 0;
  const ffc_head_config& c = h->cfg;
  const int n = in->n_rows, D = c.feat_dim;
  FFC_REQUIRE(n >= 1 && n <= c.max_rows, "ffc_head_sweep: n_rows=%d outside [1,%d]", n, c.max_rows);
  FFC_REQUIRE(in->p_f32 && in->queue_f32 && in->label && in->n_ones && in->ones_list, "ffc_head_sweep: NULL input");
  FFC_REQUIRE(out->lsum && out->osum && out->tgt && out->topv && out->topi, "ffc_head_sweep: NULL stats");
  const bool bf16 = c.precision == FFC_PREC_BF16;
  FFC_REQUIRE(!bf16 || in->queue_bf16, "ffc_head_sweep: the bf16 path needs the bf16 queue mirror");
  cudaStream_t s = (cudaStream_t)stream;
  const float* qf = in->queue_f32;
  const __nv_bfloat16* qh = (const __nv_bfloat16*)in->queue_bf16;

  const bool sv = c.loss_type == FFC_LOSS_SV;
  if (phase & 1) {
    // counts double-buffered by pass parity (see head_prep_fused_kernel)
    h->pass_parity ^= 1;
    int32_t* cur = h->counts + 2 * h->pass_parity;
    int32_t* nxt = h->counts + 2 * (h->pass_parity ^ 1);
    const int grid = std::min<int>(c.max_rows, (n + 127) & ~127);
    if (bf16)
      head_prep_fused_kernel<true><<<grid, 128, 0, s>>>(in->p_f32, h->p16, in->label, n, c.col_offset, c.q_local, D, qf, qh, in->cmask, in->ones_list,
                                                        in->n_ones, c.max_rows, nullptr, h->side_bf16, h->tcol, h->tpos, h->is_out, h->kth_shared, cur, nxt, c.margin,
                                                        out->tgt, sv ? h->thr : nullptr, use_row_map(h, n) ? h->row_map : nullptr, h->part_ctr);
    else
      head_prep_fused_kernel<false><<<grid, 128, 0, s>>>(in->p_f32, h->p16, in->label, n, c.col_offset, c.q_local, D, qf, qh, in->cmask, in->ones_list,
                                                         in->n_ones, c.max_rows, h->side_f32, nullptr, h->tcol, h->tpos, h->is_out, h->kth_shared, cur, nxt, c.margin,
                                                         out->tgt, sv ? h->thr : nullptr, nullptr, h->part_ctr);
    FFC_LAUNCH_CHECK();
    h->prepared_rows = n;
  }
  if (phase == 1) return FFC_OK;
  if (phase == 2) {
    FFC_REQUIRE(h->prepared_rows == n && n > 0, "ffc_head_sweep_prepared: ffc_head_prep was not run for these %d rows", n);
    if (sv) {
      head_thr_from_tgt_kernel<<<(n + 127) / 128, 128, 0, s>>>(out->tgt, n, c.margin, h->thr);
      FFC_LAUNCH_CHECK();
    }
  }
  h->prepared_rows = 0;

  SweepArgs a;
  memset(&a, 0, sizeof(a));
  a.P_f32 = in->p_f32;
  a.P_bf16 = h->p16;
  a.n_rows = n;
  a.D = D;
  a.is_out = h->is_out;
  a.kth_shared = h->kth_shared;
  if (use_row_map(h, n)) {      // (written by this pass's prep launch)
    a.row_map = h->row_map;
    a.n_pos_dev = h->part_ctr + 1;
  }
  a.scale = c.scale;
  a.fixed_max = fixed_max_of(c);
  a.sv = sv;
  a.k = c.topk;
  int rc;
  if (bf16 && !sv) return run_merged_sweeps(h, a, in, out, defer_reduce, s);
  // main sweep(s) over queue[0]: everything except the target column and the `ones` columns
  a.W_f32 = qf;
  a.W_bf16 = qh;
  a.n_cols = c.q_local;
  a.n_cols_dev = nullptr;
  a.tcol = h->tcol;
  a.cmask = in->cmask;
  a.thr = sv ? h->thr : nullptr;
  if ((rc = run_one_sweep(h, a, 0, 0, 0, out, c.col_offset, nullptr, s))) return rc;
  if (sv) {   // the SV hard-example threshold follows each loss's own target cosine (ffc.py:122)
    a.thr = h->thr + n;
    if ((rc = run_one_sweep(h, a, 0, 1, -1, out, c.col_offset, nullptr, s))) return rc;
  }   // (AM / Arc: both losses share the common statistics; finalize reads slot 0 for both)
  // side sweeps over the gathered `ones` rows of queue[0] and queue[1]
  a.n_cols = c.max_rows;
  a.n_cols_dev = in->n_ones;
  a.tcol = h->tpos;
  a.cmask = nullptr;
  for (int l = 0; l < 2; ++l) {
    a.W_f32 = h->side_f32 + (int64_t)l * c.max_rows * D;
    a.W_bf16 = h->side_bf16 + (int64_t)l * c.max_rows * D;
    a.thr = sv ? h->thr + (int64_t)l * n : nullptr;
    if ((rc = run_one_sweep(h, a, 1 + l, 2 + l, 1 + l, out, c.col_offset, in->ones_list, s))) return rc;
  }
  return FFC_OK;
}

extern "C" int ffc_head_sweep(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* out, void* stream) {
  return head_sweep_impl(h, in, out, false, stream);
}

extern "C" int ffc_head_prep(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* out, void* stream) {
  return head_sweep_impl(h, in, out, false, stream, 1);
}

extern "C" int ffc_head_sweep_prepared(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* out, void* stream) {
  return head_sweep_impl(h, in, out, false, stream, 2);
}

static int head_finalize_impl(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* stats, int n_ranks_topk, float* loss_out, float* dp_out,
                              void* stream);

extern "C" int ffc_head_pass_single(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* scratch, float* loss_out, float* dp_out, void* stream) {
  FFC_REQUIRE(h && in && scratch && loss_out && dp_out, "ffc_head_pass_single: NULL argument");
  int rc = head_sweep_impl(h, in, scratch, true, stream);
  if (rc) return rc;
  return head_finalize_impl(h, in, scratch, 1, loss_out, dp_out, stream);
}

extern "C" int ffc_head_finalize(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* stats, int n_ranks_topk, float* loss_out,
                                 float* dp_out, void* stream) {
  FFC_REQUIRE(h && !h->jobs_pending, "ffc_head_finalize: the last sweep was issued by ffc_head_pass_single");
  return head_finalize_impl(h, in, stats, n_ranks_topk, loss_out, dp_out, stream);
}

static FinalizeArgs make_finalize_args(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* stats, int n_ranks, float* dp_out) {
  const ffc_head_config& c = h->cfg;
  FinalizeArgs a;
  memset(&a, 0, sizeof(a));
  a.P = in->p_f32;
  a.qf = in->queue_f32;
  a.qh = (const __nv_bfloat16*)in->queue_bf16;
  a.use_bf16_rows = c.precision == FFC_PREC_BF16;
  a.label = in->label;
  a.tcol = h->tcol;
  a.tpos = h->tpos;
  a.is_out = h->is_out;
  a.counts = h->counts + 2 * h->pass_parity;
  if (stats) {
    a.lsum = stats->lsum;
    a.osum = stats->osum;
    a.tgt = stats->tgt;
    a.topv = stats->topv;
    a.topi = stats->topi;
  }
  a.n_ranks = n_ranks;
  a.n = in->n_rows;
  a.D = c.feat_dim;
  a.k = c.topk;
  a.q_local = c.q_local;
  a.col_offset = c.col_offset;
  a.loss_type = c.loss_type;
  a.scale = c.scale;
  a.margin = c.margin;
  a.fixed_max = fixed_max_of(c);
  a.cos_m = cos((double)c.margin);
  a.sin_m = sin((double)c.margin);
  a.row_loss = h->row_loss;
  a.dp = dp_out;
  if (h->want_dq) {
    a.coef_out = h->coef;
    a.nslot_out = h->nslot;
    a.wslot_out = h->wslot;
    a.wrow_out = h->wrow;
  }
  return a;
}

static int head_finalize_impl(ffc_head_t* h, const ffc_head_pass* in, const ffc_head_stats* stats, int n_ranks_topk, float* loss_out, float* dp_out,
                              void* stream) {
  FFC_REQUIRE(h && in && stats && loss_out && dp_out, "ffc_head_finalize: NULL argument");
  FFC_REQUIRE(n_ranks_topk >= 1, "ffc_head_finalize: n_ranks_topk must be >= 1");
  cudaStream_t s = (cudaStream_t)stream;
  const FinalizeArgs a = make_finalize_args(h, in, stats, n_ranks_topk, dp_out);
  if (h->jobs_pending) {       // one-GPU fast path: the sweep left its partials for the fused reduce + finalize
    FFC_REQUIRE(n_ranks_topk == 1, "fused finalize is single-rank");
    h->jobs_pending = 0;
    head_finalize_fused_kernel<false><<<(a.n + FR - 1) / FR, 128, 0, s>>>(*h->jobs, a, nullptr, 0);
    FFC_LAUNCH_CHECK();
  } else {
    head_row_coef_kernel<<<(a.n + 127) / 128, 128, 0, s>>>(a, h->coef, h->nslot, h->wslot, h->wrow);
    FFC_LAUNCH_CHECK();
    head_finalize_kernel<<<a.n, 128, 0, s>>>(a, h->coef, h->nslot, h->wslot, h->wrow);
    FFC_LAUNCH_CHECK();
  }
  head_loss_sum_kernel<<<1, 1024, 0, s>>>(h->row_loss, a.n, loss_out);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

// ---- sharded head: per-rank record out of the sweep, finalize from the gathered records ----
// Record exchange by peer stores (sharded head, ranks whose record buffers are peer-mapped): copies this rank's record of the pass just
// swept into EVERY rank's gathered buffer -- the 8 scalars of every row always, the top-k candidate slots (88 % of a record at k = 10)
// only for hard-negative-only rows, the only rows whose candidates the fused finalize reads.  An all-gather cannot trim by content; at C3
// (no such rows) this is 0.26 MB per pass and rank instead of 2.2 MB.
__global__ void __launch_bounds__(256) head_push_record_kernel(const float* __restrict__ rec, int n, int k, const uint8_t* __restrict__ is_out,
                                                               float* const* __restrict__ peers, int64_t dst_off, int n_ranks) {
  const int64_t n_scalar4 = 2 * (int64_t)n;                       // 8 n words as float4 (8 n is a multiple of 4)
  const int64_t n_top = 6 * (int64_t)n * k;                       // [3][n][k] values, then [3][n][k] columns
  const int64_t total = n_scalar4 + n_top;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    if (e < n_scalar4) {
      const float4 v = reinterpret_cast<const float4*>(rec)[e];
      for (int r = 0; r < n_ranks; ++r) reinterpret_cast<float4*>(peers[r] + dst_off)[e] = v;
    } else {
      const int64_t t = e - n_scalar4;
      const int row = (int)((t / k) % n);
      if (!is_out[row]) continue;
      const float v = rec[8 * (int64_t)n + t];
      for (int r = 0; r < n_ranks; ++r) peers[r][dst_off + 8 * (int64_t)n + t] = v;
    }
  }
  __threadfence_system();      // visible system-wide before the kernel counts as finished; the flag follows in ffc_peer_barrier
}

extern "C" int ffc_head_push_record(ffc_head_t* h, int n_rows, const float* record_dev, float* const* peer_ptrs_dev, int64_t dst_offset_words, int n_ranks,
                                    void* stream) {
  FFC_REQUIRE(h && record_dev && peer_ptrs_dev && n_rows >= 1 && n_rows <= h->cfg.max_rows && n_ranks >= 1 && n_ranks <= 64 && dst_offset_words >= 0 &&
                  dst_offset_words % 4 == 0,
              "ffc_head_push_record: bad arguments");
  const int64_t total = 2 * (int64_t)n_rows + 6 * (int64_t)n_rows * h->cfg.topk;
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div64(total, 256), 148 * 2));
  head_push_record_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(record_dev, n_rows, h->cfg.topk, h->is_out, peer_ptrs_dev, dst_offset_words, n_ranks);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

extern "C" int ffc_head_record_words(const ffc_head_config* cfg, int n_rows, int64_t* words_out) {
  FFC_REQUIRE(cfg && words_out && n_rows >= 0, "ffc_head_record_words: bad arguments");
  *words_out = record_words(n_rows, cfg->topk);
  return FFC_OK;
}

extern "C" int ffc_head_sweep_record(ffc_head_t* h, const ffc_head_pass* in, void* record_out, void* stream) {
  FFC_REQUIRE(h && in && record_out, "ffc_head_sweep_record: NULL argument");
  FFC_REQUIRE(h->cfg.precision == FFC_PREC_BF16 && h->cfg.loss_type != FFC_LOSS_SV, "ffc_head_sweep_record: bf16 AM / Arc only");
  const int n = in->n_rows, k = h->cfg.topk;
  float* rec = (float*)record_out;
  ffc_head_stats st;
  memset(&st, 0, sizeof(st));
  st.lsum = rec;                       // unused by the deferred path, but head_sweep_impl wants non-NULL statistics
  st.osum = h->o_part;
  st.tgt = rec + 4 * (int64_t)n;       // the prep kernel writes the target cosines straight into the record
  st.topv = rec + 8 * (int64_t)n;
  st.topi = (int32_t*)(rec + 8 * (int64_t)n + 3 * (int64_t)n * k);
  int rc = head_sweep_impl(h, in, &st, true, stream);
  if (rc) return rc;
  FFC_REQUIRE(h->jobs_pending, "ffc_head_sweep_record: merged sweep path not taken");
  head_reduce_scalars_kernel<<<(3 * n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*h->jobs, n, k, h->is_out, rec);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

extern "C" int ffc_head_finalize_gathered(ffc_head_t* h, const ffc_head_pass* in, const void* records, int n_ranks, int64_t record_stride_words,
                                          float* loss_out, float* dp_out, void* stream) {
  return ffc_head_finalize_gathered_ex(h, in, records, n_ranks, record_stride_words, nullptr, loss_out, dp_out, stream);
}

extern "C" int ffc_head_finalize_gathered_ex(ffc_head_t* h, const ffc_head_pass* in, const void* records, int n_ranks, int64_t record_stride_words,
                                             const ffc_head_finalize_opts* opts, float* loss_out, float* dp_out, void* stream) {
  FFC_REQUIRE(h && in && records && loss_out && n_ranks >= 1, "ffc_head_finalize_gathered: bad arguments");
  FFC_REQUIRE(dp_out || (opts && opts->dp_peer), "ffc_head_finalize_gathered: neither dp_out nor peer staging buffers given");
  FFC_REQUIRE(h->jobs_pending, "ffc_head_finalize_gathered: no ffc_head_sweep_record pending");
  FFC_REQUIRE(record_stride_words >= record_words(in->n_rows, h->cfg.topk), "ffc_head_finalize_gathered: record stride too small");
  cudaStream_t s = (cudaStream_t)stream;
  FinalizeArgs a = make_finalize_args(h, in, nullptr, n_ranks, dp_out);
  if (opts) {
    FFC_REQUIRE(!opts->overlay_map || (opts->overlay_g && opts->overlay_undo), "ffc_head_finalize_gathered_ex: overlay map without its row tables");
    FFC_REQUIRE(!opts->dp_peer || opts->dp_rows_per_rank >= 1, "ffc_head_finalize_gathered_ex: dp_rows_per_rank must be >= 1");
    a.ovl_map = opts->overlay_map;
    a.ovl_g = opts->overlay_g;
    a.ovl_undo = opts->overlay_undo;
    a.dp_peer = opts->dp_peer;
    a.dp_rows_per_rank = opts->dp_rows_per_rank;
    a.dp_slot_off = opts->dp_slot_offset;
  }
  h->jobs_pending = 0;
  head_finalize_fused_kernel<true><<<(a.n + FR - 1) / FR, 128, 0, s>>>(*h->jobs, a, (const float*)records, record_stride_words);
  FFC_LAUNCH_CHECK();
  head_loss_sum_kernel<<<1, 1024, 0, s>>>(h->row_loss, a.n, loss_out);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

extern "C" int ffc_head_set_timing(ffc_head_t* h, int enable) {
  FFC_REQUIRE(h != nullptr, "ffc_head_set_timing: NULL handle");
  h->timing = enable ? 1 : 0;
  h->ev_used = 0;
  return FFC_OK;
}

extern "C" int ffc_head_get_timing(ffc_head_t* h, double* total_ms_out, int64_t* launches_out) {
  FFC_REQUIRE(h && total_ms_out && launches_out, "ffc_head_get_timing: NULL argument");
  double tot = 0.0;
  for (size_t i = 0; i + 1 < h->ev_used; i += 2) {
    FFC_CUDA(cudaEventSynchronize((*h->ev)[i + 1]));
    float ms = 0.f;
    FFC_CUDA(cudaEventElapsedTime(&ms, (*h->ev)[i], (*h->ev)[i + 1]));
    tot += ms;
  }
  *total_ms_out = tot;
  *launches_out = (int64_t)(h->ev_used / 2);
  return FFC_OK;
}

// ------------------------------------------------------------------------------------------------
// Optional mode: dLoss/dQueue (the reference keeps `queue` a no-grad buffer, ffc.py:29; north_star asks for "dQueue where the queue
// is trainable").  For the pass just finalized, with z_ij = s cos_ij (j != t_i), L_l,i the softmax denominators and
// a_l,i = s / (n_pos L_l,i) (finalize's cO), every queue row gets
//     dqueue[0][j] = sum_i (a_1i + a_2i) p~_ij p_i                                  for j outside C u T   (the bulk: Q x n x D)
// -- the SAME sweep kernel with the roles swapped: the queue rows are the "probe rows", the n probe embeddings the columns, GEMM-1
// recomputes the cosines from the bf16 probe rows and GEMM-2 accumulates the probe rows scaled by their coefficient (W2 operand),
// so dqueue[0] comes out of TMEM row tile by row tile: 4 n Q D more FLOPs per pass, no B x Q matrix.  The <= 2n "special" slots --
// targets T (the margin changes their coefficient) and `ones` C (losses 1 / 2 read different rows) -- are recomputed exactly by a
// small SIMT kernel and overwritten; the hard-negative term adds w_neg p_i to the <= 2k rows each outlier row selected.
// SV: the hardness test cos_ij > thr_l,i is per probe row, i.e. per COLUMN of the swapped sweep, and the two losses' p~ differ where
// their thresholds do.  The sweep's DQ_SV mode forms the combined weight sum_l a_l,i p~_l,ij h'_l,ij (h' = 1.2 on hard columns, else
// 1; z = 1.2 cos + 0.2 there) in its epilogue from per-column scalars and accumulates the raw probe rows.
// Check mode (FFC_PREC_FP32): one SIMT kernel per queue slot with fp64 dots and sums in a fixed order computes every row -- bulk,
// targets and `ones` alike -- and a one-owner-per-feature kernel adds the hard negatives: no atomics, bit-identical from run to run.
// ------------------------------------------------------------------------------------------------
namespace ffc {

__global__ void __launch_bounds__(128) dq_scale_probe_kernel(const __nv_bfloat16* __restrict__ p16, const float* __restrict__ coef, const uint8_t* __restrict__ is_out,
                                                             int n, int D, __nv_bfloat16* __restrict__ pc16) {
  const int i = blockIdx.x;
  const float c = is_out[i] ? 0.f : coef[0 * n + i] + coef[1 * n + i];
  for (int d = threadIdx.x; d < D; d += blockDim.x) pc16[(int64_t)i * D + d] = __float2bfloat16(c * __bfloat162float(p16[(int64_t)i * D + d]));
}

// per probe row: (thr_1, thr_2, a_1, a_2), the coefficients zero on hard-negative-only rows (their term is dq_hard_neg_kernel's)
__global__ void __launch_bounds__(128) dq_sv_cols_kernel(const float* __restrict__ thr, const float* __restrict__ coef, const uint8_t* __restrict__ is_out, int n,
                                                         float4* __restrict__ col) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const bool o = is_out[i];
  col[i] = make_float4(thr[i], thr[n + i], o ? 0.f : coef[0 * n + i], o ? 0.f : coef[1 * n + i]);
}

// p~ h' of one non-target cosine: SV (thr != NULL) applies the hard-example transform above the row's threshold
__device__ __forceinline__ float dq_pt(float dot, float a2, float b2, float th) {
  const bool m = dot > th;
  return exp2f(fmaf(m ? fmaf(SV_T, dot, SV_T - 1.f) : dot, a2, -b2)) * (m ? SV_T : 1.f);
}

// one block per candidate special slot: blocks [0, max_rows) take ones_list[b] (if b < n_ones), blocks [max_rows, max_rows + n) the
// target of probe row b - max_rows (if it is local, not in C -- those are the first kind -- and not claimed by another row's block).
// SV: `thr` [2][n] holds the per-row thresholds of the two losses.
template <bool SV>
__global__ void __launch_bounds__(256) dq_special_rows_kernel(const __nv_bfloat16* __restrict__ p16, const __nv_bfloat16* __restrict__ qh, int64_t q_local, int D, int n,
                                                              int max_rows, const int32_t* __restrict__ ones_list, const int32_t* __restrict__ n_ones_p,
                                                              const uint32_t* __restrict__ cmask_unused, const int32_t* __restrict__ tcol,
                                                              const int32_t* __restrict__ tpos, const uint8_t* __restrict__ is_out, const float* __restrict__ coef,
                                                              const float* __restrict__ thr, float a2, float b2, int32_t* __restrict__ claim, int32_t epoch,
                                                              float* __restrict__ dq) {
  extern __shared__ float sm[];          // [D] queue row, [n] coefficients
  float* s_q = sm;
  float* s_c = sm + D;
  const int b = blockIdx.x;
  int slot;
  bool in_c;
  if (b < max_rows) {
    if (b >= *n_ones_p) return;
    slot = ones_list[b];
    in_c = true;
  } else {
    const int i = b - max_rows;
    if (i >= n || is_out[i] || tcol[i] < 0 || tpos[i] >= 0) return;      // tpos >= 0: the target is in C
    slot = tcol[i];
    in_c = false;
    __shared__ int mine;
    if (threadIdx.x == 0) mine = atomicExch(&claim[slot], epoch) != epoch;
    __syncthreads();
    if (!mine) return;
  }
  for (int r = 0; r < (in_c ? 2 : 1); ++r) {
    const __nv_bfloat16* qrow = qh + ((int64_t)r * q_local + slot) * D;
    __syncthreads();
    for (int d = threadIdx.x; d < D; d += blockDim.x) s_q[d] = __bfloat162float(qrow[d]);
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      float c = 0.f;
      if (!is_out[i]) {
        const bool is_t = tcol[i] == slot;
        if (is_t) {
          // the target column: d/dcos of the margined logit, from finalize (cT); loss 2 reads queue[1] iff the slot is in C
          if (r == 0) c += coef[2 * n + i];
          if (r == (in_c ? 1 : 0)) c += coef[3 * n + i];
        } else {
          const __nv_bfloat162* pr = reinterpret_cast<const __nv_bfloat162*>(p16 + (int64_t)i * D);
          float dot = 0.f;
          for (int d = 0; d < D; d += 2) {
            const float2 v = __bfloat1622float2(pr[d >> 1]);
            dot = fmaf(v.x, s_q[d], dot);
            dot = fmaf(v.y, s_q[d + 1], dot);
          }
          if (SV) {
            c = in_c ? coef[r * n + i] * dq_pt(dot, a2, b2, thr[r * n + i])
                     : coef[0 * n + i] * dq_pt(dot, a2, b2, thr[i]) + coef[1 * n + i] * dq_pt(dot, a2, b2, thr[n + i]);
          } else {
            const float pt = exp2f(fmaf(dot, a2, -b2));
            c = in_c ? coef[r * n + i] * pt : (coef[0 * n + i] + coef[1 * n + i]) * pt;
          }
        }
      }
      s_c[i] = c;
    }
    __syncthreads();
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
      float acc = 0.f;
      for (int i = 0; i < n; ++i) acc = fmaf(s_c[i], __bfloat162float(p16[(int64_t)i * D + d]), acc);
      dq[((int64_t)r * q_local + slot) * D + d] = acc;
    }
  }
}

// hard negatives (ffc.py:86-92): outlier row i adds w_neg p_i to the prototype rows finalize selected for it
__global__ void __launch_bounds__(128) dq_hard_neg_kernel(const __nv_bfloat16* __restrict__ p16, const uint8_t* __restrict__ is_out, const float* __restrict__ coef,
                                                          const int32_t* __restrict__ nslot, const int32_t* __restrict__ wslot, const uint8_t* __restrict__ wrow, int n,
                                                          int D, int64_t q_local, int64_t col_offset, float* __restrict__ dq) {
  const int i = blockIdx.x;
  if (!is_out[i]) return;
  const float w = coef[0 * n + i];
  const int nw = nslot[i];
  for (int x = 0; x < nw; ++x) {
    const int64_t loc = (int64_t)wslot[(int64_t)i * 2 * KMAX + x] - col_offset;
    if (loc < 0 || loc >= q_local) continue;
    float* dst = dq + ((int64_t)wrow[(int64_t)i * 2 * KMAX + x] * q_local + loc) * D;
    for (int d = threadIdx.x; d < D; d += blockDim.x) atomicAdd(dst + d, w * __bfloat162float(p16[(int64_t)i * D + d]));
  }
}

// Check mode: one block per local slot j writes dqueue[0][j] and dqueue[1][j] whole.  Per probe row i (fp64 on the fp32 inputs):
//   target of i (tcol[i] == j):  d/dcos of the margined logit from finalize (cT), loss 2's on queue[1] iff j is in C
//   otherwise:                   a_l,i p~_l,ij h'_l,ij, with loss 2 reading queue[1][j] iff j is in C (and nothing reading it else)
// hard-negative-only rows contribute nothing here (dq_hard_neg_f32_kernel).  Sums over i run in index order.
__global__ void __launch_bounds__(128) dq_rows_f32_kernel(const float* __restrict__ P, const float* __restrict__ qf, int64_t q_local, int D, int n,
                                                          const uint32_t* __restrict__ cmask, const int32_t* __restrict__ tcol, const uint8_t* __restrict__ is_out,
                                                          const float* __restrict__ coef, const float* __restrict__ thr, double s, double M,
                                                          float* __restrict__ dq) {
  extern __shared__ double smd[];        // [2][D] queue rows, [2][n] coefficients
  double* s_q = smd;
  double* s_c = smd + 2 * D;
  const int64_t j = blockIdx.x;
  const bool in_c = cmask && ((cmask[j >> 5] >> (j & 31)) & 1u);
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    s_q[d] = qf[j * D + d];
    s_q[D + d] = qf[(q_local + j) * D + d];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    double c0 = 0.0, c1 = 0.0;      // coefficients of p_i in dqueue[0][j] and dqueue[1][j]
    if (!is_out[i]) {
      if (tcol[i] == j) {
        c0 = coef[2 * n + i];
        if (in_c) c1 = coef[3 * n + i]; else c0 += coef[3 * n + i];
      } else {
        const float* pr = P + (int64_t)i * D;
        double dot[2] = {0.0, 0.0};
        for (int d = 0; d < D; ++d) dot[0] += (double)pr[d] * s_q[d];
        if (in_c)
          for (int d = 0; d < D; ++d) dot[1] += (double)pr[d] * s_q[D + d];
        else
          dot[1] = dot[0];
        double g[2];
        for (int l = 0; l < 2; ++l) {
          const bool hard = thr && dot[l] > (double)thr[l * n + i];
          const double z = hard ? (double)SV_T * dot[l] + (double)SV_T - 1.0 : dot[l];
          g[l] = (double)coef[l * n + i] * exp(s * z - M) * (hard ? (double)SV_T : 1.0);
        }
        c0 = g[0];
        if (in_c) c1 = g[1]; else c0 += g[1];
      }
    }
    s_c[i] = c0;
    s_c[n + i] = c1;
  }
  __syncthreads();
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    double a0 = 0.0, a1 = 0.0;
    for (int i = 0; i < n; ++i) {
      const double pv = P[(int64_t)i * D + d];
      a0 += s_c[i] * pv;
      a1 += s_c[n + i] * pv;
    }
    dq[j * D + d] = (float)a0;
    dq[(q_local + j) * D + d] = (float)a1;
  }
}

// Check mode, hard negatives: a thread owns feature d of every destination row and walks the outlier rows and their selections in
// order -- deterministic where dq_hard_neg_kernel's atomics are not
__global__ void __launch_bounds__(128) dq_hard_neg_f32_kernel(const float* __restrict__ P, const uint8_t* __restrict__ is_out, const float* __restrict__ coef,
                                                              const int32_t* __restrict__ nslot, const int32_t* __restrict__ wslot, const uint8_t* __restrict__ wrow,
                                                              int n, int D, int64_t q_local, int64_t col_offset, float* __restrict__ dq) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  for (int i = 0; i < n; ++i) {
    if (!is_out[i]) continue;
    const float w = coef[0 * n + i] * P[(int64_t)i * D + d];
    for (int x = 0; x < nslot[i]; ++x) {
      const int64_t loc = (int64_t)wslot[(int64_t)i * 2 * KMAX + x] - col_offset;
      if (loc >= 0 && loc < q_local) dq[((int64_t)wrow[(int64_t)i * 2 * KMAX + x] * q_local + loc) * D + d] += w;
    }
  }
}

}  // namespace ffc

extern "C" int ffc_head_set_dqueue(ffc_head_t* h, int enable) {
  FFC_REQUIRE(h != nullptr, "ffc_head_set_dqueue: NULL handle");
  // (check mode needs no scratch: dq_rows_f32_kernel writes every row)
  if (enable && h->cfg.precision == FFC_PREC_BF16 && !h->dq_claim) {
    const int64_t R = h->cfg.max_rows, D = h->cfg.feat_dim, Q = h->cfg.q_local;
    if (h->cfg.loss_type == FFC_LOSS_SV)
      FFC_CUDA(cudaMalloc(&h->dq_col, R * sizeof(float4)));
    else
      FFC_CUDA(cudaMalloc(&h->pc16, R * D * sizeof(__nv_bfloat16)));
    FFC_CUDA(cudaMalloc(&h->dq_l, Q * sizeof(float)));
    FFC_CUDA(cudaMalloc(&h->dq_tv, Q * sizeof(float)));
    FFC_CUDA(cudaMalloc(&h->dq_ti, Q * sizeof(int32_t)));
    FFC_CUDA(cudaMalloc(&h->dq_claim, Q * sizeof(int32_t)));
    FFC_CUDA(cudaMemset(h->dq_claim, 0, Q * sizeof(int32_t)));
  }
  h->want_dq = enable ? 1 : 0;
  return FFC_OK;
}

template <bool SV>
static int launch_dq_special_rows(ffc_head_t* h, const ffc_head_pass* in, const __nv_bfloat16* qh, size_t smem, float* dqueue_out, cudaStream_t s) {
  static bool attr_set = false;
  if (!attr_set) {
    FFC_CUDA(cudaFuncSetAttribute(dq_special_rows_kernel<SV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_set = true;
  }
  const ffc_head_config& c = h->cfg;
  dq_special_rows_kernel<SV><<<c.max_rows + in->n_rows, 256, smem, s>>>(h->p16, qh, c.q_local, c.feat_dim, in->n_rows, c.max_rows, in->ones_list, in->n_ones, in->cmask,
                                                                        h->tcol, h->tpos, h->is_out, h->coef, SV ? h->thr : nullptr, c.scale * 1.4426950408889634f,
                                                                        fixed_max_of(c) * 1.4426950408889634f, h->dq_claim, h->dq_epoch, dqueue_out);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

extern "C" int ffc_head_dqueue(ffc_head_t* h, const ffc_head_pass* in, float* dqueue_out, void* stream) {
  FFC_REQUIRE(h && in && dqueue_out, "ffc_head_dqueue: NULL argument");
  FFC_REQUIRE(h->want_dq, "ffc_head_dqueue: enable the mode with ffc_head_set_dqueue before the pass");
  const ffc_head_config& c = h->cfg;
  const int n = in->n_rows, D = c.feat_dim;
  const bool bf16 = c.precision == FFC_PREC_BF16, sv = c.loss_type == FFC_LOSS_SV;
  FFC_REQUIRE(n >= 1 && n <= c.max_rows && in->ones_list && in->n_ones, "ffc_head_dqueue: bad pass description");
  FFC_REQUIRE(bf16 ? in->queue_bf16 != nullptr : (in->p_f32 && in->queue_f32), "ffc_head_dqueue: %s", bf16 ? "the bf16 head needs the bf16 queue mirror"
                                                                                                           : "check mode needs p_f32 and queue_f32");
  FFC_REQUIRE(c.q_local < ((int64_t)1 << 31) / 2, "ffc_head_dqueue: shard too large");
  cudaStream_t s = (cudaStream_t)stream;
  if (!bf16) {
    const size_t smem = (size_t)(2 * D + 2 * n) * sizeof(double);
    FFC_REQUIRE(smem <= 200 * 1024, "ffc_head_dqueue: %d rows exceed the check-mode kernel's shared memory", n);
    static bool attr_set = false;
    if (!attr_set) {
      FFC_CUDA(cudaFuncSetAttribute(dq_rows_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attr_set = true;
    }
    dq_rows_f32_kernel<<<(unsigned)c.q_local, 128, smem, s>>>(in->p_f32, in->queue_f32, c.q_local, D, n, in->cmask, h->tcol, h->is_out, h->coef, sv ? h->thr : nullptr,
                                                              (double)c.scale, (double)fixed_max_of(c), dqueue_out);
    FFC_LAUNCH_CHECK();
    dq_hard_neg_f32_kernel<<<(D + 127) / 128, 128, 0, s>>>(in->p_f32, h->is_out, h->coef, h->nslot, h->wslot, h->wrow, n, D, c.q_local, c.col_offset, dqueue_out);
    FFC_LAUNCH_CHECK();
    return FFC_OK;
  }
  const size_t smem = (size_t)(D + n) * sizeof(float);
  FFC_REQUIRE(smem <= 200 * 1024, "ffc_head_dqueue: %d rows exceed the special-row kernel's shared memory", n);
  const __nv_bfloat16* qh = (const __nv_bfloat16*)in->queue_bf16;
  if (sv) {
    dq_sv_cols_kernel<<<(n + 127) / 128, 128, 0, s>>>(h->thr, h->coef, h->is_out, n, h->dq_col);
  } else {
    dq_scale_probe_kernel<<<n, 128, 0, s>>>(h->p16, h->coef, h->is_out, n, D, h->pc16);
  }
  FFC_LAUNCH_CHECK();
  // the swapped sweep: "probe rows" = the queue rows of queue[0], columns = the n probe embeddings
  SweepArgs a;
  memset(&a, 0, sizeof(a));
  a.P_bf16 = qh;
  a.n_rows = (int)c.q_local;
  a.D = D;
  a.W_bf16 = h->p16;
  a.W2_bf16 = sv ? nullptr : h->pc16;       // SV: the coefficients are in the epilogue's weights, GEMM-2 sums the raw probe rows
  a.dq_col = sv ? h->dq_col : nullptr;
  a.force_pair = 1;
  a.n_cols = n;
  a.kth_shared = h->kth_shared;
  a.scale = c.scale;
  a.fixed_max = fixed_max_of(c);
  a.k = 1;
  a.n_chunks = 1;
  a.l_part = h->dq_l;
  a.o_part = dqueue_out;
  a.topv_part = h->dq_tv;
  a.topi_part = h->dq_ti;
  int rc = launch_sweeps_sm100(h->sm100, &a, 1, s);
  if (rc) return rc;
  FFC_CUDA(cudaMemsetAsync(dqueue_out + c.q_local * D, 0, (size_t)c.q_local * D * sizeof(float), s));
  h->dq_epoch += 1;
  if ((rc = sv ? launch_dq_special_rows<true>(h, in, qh, smem, dqueue_out, s) : launch_dq_special_rows<false>(h, in, qh, smem, dqueue_out, s))) return rc;
  dq_hard_neg_kernel<<<n, 128, 0, s>>>(h->p16, h->is_out, h->coef, h->nslot, h->wslot, h->wrow, n, D, c.q_local, c.col_offset, dqueue_out);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

// ------------------------------------------------------------------------------------------------
// 1:N identification against queue[0] (identify_sm100.cu)
// ------------------------------------------------------------------------------------------------
extern "C" int ffc_identify_workspace_bytes(ffc_head_t* h, int n, int k, int64_t* bytes_out) {
  FFC_REQUIRE(n >= 1 && n <= FFC_IDENTIFY_MAX_ROWS, "ffc_identify_workspace_bytes: n=%d rows outside [1, %d]", n, FFC_IDENTIFY_MAX_ROWS);
  FFC_REQUIRE(k >= 1 && k <= KMAX, "ffc_identify_workspace_bytes: k=%d outside [1, %d]", k, KMAX);
  FFC_REQUIRE(h && bytes_out, "ffc_identify_workspace_bytes: NULL argument");
  *bytes_out = identify_workspace_bytes(h->cfg.precision == FFC_PREC_BF16, n, k, h->cfg.q_local);
  return FFC_OK;
}

extern "C" int ffc_identify(ffc_head_t* h, const ffc_lru_t* lru, const float* x_f32, int n, int k, const float* queue_f32, const void* queue_bf16,
                            void* workspace, int64_t workspace_bytes, float* score_out, int64_t* label_out, int32_t* slot_out, void* stream) {
  FFC_REQUIRE(n >= 1 && n <= FFC_IDENTIFY_MAX_ROWS, "ffc_identify: n=%d rows outside [1, %d] (split larger inputs)", n, FFC_IDENTIFY_MAX_ROWS);
  FFC_REQUIRE(k >= 1 && k <= KMAX, "ffc_identify: k=%d outside [1, %d]", k, KMAX);
  FFC_REQUIRE(h && lru, "ffc_identify: NULL head or LRU handle");
  FFC_REQUIRE(x_f32 && queue_f32 && workspace && score_out && label_out && slot_out, "ffc_identify: NULL device pointer");
  const ffc_head_config& c = h->cfg;
  const bool bf16 = c.precision == FFC_PREC_BF16;
  FFC_REQUIRE(!bf16 || queue_bf16, "ffc_identify: the bf16 path needs the bf16 queue mirror");
  const int64_t need = identify_workspace_bytes(bf16, n, k, c.q_local);
  FFC_REQUIRE(workspace_bytes >= need, "ffc_identify: workspace of %lld bytes, %lld needed", (long long)workspace_bytes, (long long)need);
  const int32_t* cur_idx = nullptr;
  const int64_t* slot_key = nullptr;
  int64_t cap = 0;
  int rc = lru_device_state(lru, &cur_idx, &slot_key, &cap);
  if (rc) return rc;
  FFC_REQUIRE(cap <= c.q_local, "ffc_identify: LRU capacity %lld exceeds the head's %lld queue slots", (long long)cap, (long long)c.q_local);
  IdentifyArgs a;
  a.x = x_f32;
  a.queue_f32 = queue_f32;
  a.queue_bf16 = bf16 ? queue_bf16 : nullptr;
  a.q_local = c.q_local;
  a.col_offset = c.col_offset;
  a.cur_idx_dev = cur_idx;
  a.slot_key = slot_key;
  a.n_rows = n;
  a.D = c.feat_dim;
  a.k = k;
  a.workspace = workspace;
  a.score_out = score_out;
  a.label_out = label_out;
  a.slot_out = slot_out;
  return launch_identify(h->sm100, a, (cudaStream_t)stream);
}
