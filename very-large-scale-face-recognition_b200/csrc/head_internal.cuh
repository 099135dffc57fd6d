// Internal interfaces of the fused margin-softmax head (shared by the check-mode SIMT sweep, the
// tcgen05 sweep, the partial reduce and finalize).
#pragma once
#include "ffc_common.cuh"

namespace ffc {

constexpr int KMAX = FFC_TOPK_MAX;
constexpr float SV_T = 1.2f;  // ffc.py:47 mask_svfc

// One sweep = one pass over a [n_cols, D] weight matrix for all probe rows, producing per
// (column-chunk, row) partials.  Excluded per row: column tcol[row] (the target) and every column
// whose bit is set in cmask (main sweep only).  p~ = exp(scale*z(cos) - M), z(cos) = cos, or
// SV_T*cos + SV_T - 1 where cos > thr[row] (SV only; thr = +inf otherwise).
struct SweepArgs {
  const float* W_f32;            // [n_cols, D] (check mode)
  const __nv_bfloat16* W_bf16;   // [n_cols, D] (tensor-core mode)
  const __nv_bfloat16* W2_bf16;  // optional: the matrix GEMM-2 accumulates (O += p~ . W2) when it is not W itself -- the queue-gradient
                                 // sweep reads the probe rows for the cosines and the coefficient-scaled probe rows for the sum.  CTA-pair kernel only.
  int force_pair;                // run on the CTA-pair kernel whatever D is
  const float* P_f32;            // [n_rows, D]
  const __nv_bfloat16* P_bf16;   // [n_rows, D]
  int64_t n_cols;                // host-side bound on the number of columns
  const int32_t* n_cols_dev;     // optional device-side actual count (<= n_cols); NULL -> n_cols
  int n_rows;
  int D;
  const int32_t* tcol;           // [n_rows] excluded column or -1
  const uint32_t* cmask;         // bit per column or NULL
  const float* thr;              // [n_rows] or NULL (=> +inf)
  const uint8_t* is_out;         // [n_rows] 1 if the row takes part in the hard-negative top-k
  const int32_t* row_map;        // optional [n_rows]: sweep position -> probe row, hard-negative-only rows last (CTA-pair tcgen05 kernel; NULL = identity)
  const int32_t* n_pos_dev;      // ... and the number of rows in front of them (device side)
  int32_t* kth_shared;           // [n_rows] zero-initialised scratch: threshold shared by the column chunks (tcgen05 path; never NULL there)
  float scale;                   // s
  float fixed_max;               // M
  int sv;                        // SV transform enabled
  int k;                         // top-k size
  int n_chunks;                  // column chunks (partials per row)
  // partial outputs
  float* l_part;                 // [n_chunks][n_rows]
  float* o_part;                 // [n_chunks][n_rows][D]
  float* topv_part;              // [n_chunks][n_rows][k]   descending, -inf padded
  int32_t* topi_part;            // [n_chunks][n_rows][k]   LOCAL column indices
  const float4* dq_col;          // optional: the SV queue-gradient sweep's per-column (thr_1, thr_2, a_1, a_2); selects that kernel mode.  CTA-pair kernel only.
};

int launch_sweep_simt(const SweepArgs& a, cudaStream_t s);
// tcgen05 path (head_sm100.cu).  `cache_slot` selects one of the handle's tensor-map cache entries.
struct Sm100Cache;
Sm100Cache* sm100_cache_create();
void sm100_cache_destroy(Sm100Cache*);
int launch_sweep_sm100(Sm100Cache* cache, int cache_slot, const SweepArgs& a, cudaStream_t s);
// up to three sweeps that share the probe rows in ONE launch (main + the two side sweeps)
int launch_sweeps_sm100(Sm100Cache* cache, const SweepArgs* sweeps, int n_sweeps, cudaStream_t s);
int sm100_pick_chunks(int n_rows, int64_t n_cols, int D, int chunk_cap);   // chunk_cap: most column chunks the partial workspace holds

// sorted (descending) insertion into a k-entry list held in registers / local arrays
template <int K>
__device__ __forceinline__ void topk_insert(float (&v)[K], int32_t (&ix)[K], int k, float x, int32_t xi) {
#pragma unroll
  for (int r = 0; r < K; ++r) {
    if (r < k && x > v[r]) {
      const float tv = v[r];
      const int32_t ti = ix[r];
      v[r] = x;
      ix[r] = xi;
      x = tv;
      xi = ti;
    }
  }
}

}  // namespace ffc
