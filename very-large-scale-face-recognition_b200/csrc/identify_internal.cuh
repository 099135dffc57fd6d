// Internal interface of the identification search (identify_sm100.cu), called by ffc_identify (head.cu).
#pragma once
#include "head_internal.cuh"

namespace ffc {

struct IdentifyArgs {
  const float* x;               // [n_rows, D] unit query rows
  const float* queue_f32;       // [q_local, D] queue[0] (rescoring; check mode: also the search)
  const void* queue_bf16;       // [q_local, D] bf16 mirror of queue[0]: tensor-core search; NULL = check mode
  int64_t q_local;
  int64_t col_offset;
  const int32_t* cur_idx_dev;   // resident slots [0, *cur_idx_dev)
  const int64_t* slot_key;      // [q_local] key of each slot
  int n_rows, D, k;
  void* workspace;              // identify_workspace_bytes()
  float* score_out;
  int64_t* label_out;
  int32_t* slot_out;
};

int identify_chunks(bool bf16, int n_rows, int64_t q_local);
int64_t identify_workspace_bytes(bool bf16, int n_rows, int k, int64_t q_local);
// launches per call: bf16: search + merge (after a memset of the shared thresholds); check mode: search + merge
int launch_identify(Sm100Cache* cache, const IdentifyArgs& a, cudaStream_t s);

// the LRU's device-side state (lru.cu): cur_idx, slot_key[], capacity
int lru_device_state(const ffc_lru_t* h, const int32_t** cur_idx_dev, const int64_t** slot_key, int64_t* capacity);

}  // namespace ffc
