// Device-resident LRU id->slot cache with an undo journal (replaces /root/reference lru.py:21-255
// and the bookkeeping loops ffc.py:162-177 / ffc.py:214-235).
//
// Layout in HBM (capacity = Q slots):
//   ht_key[T] int64 / ht_slot[T] int32   open-addressing table, T = pow2 >= 4Q, probed in aligned
//                                        32-cell windows by one warp (ballot match / ballot empty);
//                                        deletions leave tombstones, the table is rebuilt when the
//                                        host-side upper bound of used cells passes T/2.
//   slot_key[Q] int64, last_pos[Q] int64 authoritative per-slot state.
//   ring[RC] int32 (x2, RC = pow2 >= 4Q) log-structured recency: every access appends its slot at
//                                        absolute position head++; a record is live iff
//                                        last_pos[slot] == position.  LRU order == live records in
//                                        ring order, so "the M least recently used entries" is a
//                                        coalesced window scan from `tail`, not a pointer chase.
//   journal[J]                           one entry per journaled access (try_get) for exact undo.
//
// One batch (<= 1024 keys) is resolved by ONE CTA: the reference semantics are sequential in batch
// order (an entry resident at batch start can be evicted by an earlier miss of the same batch and
// re-inserted elsewhere), so the CTA builds the "local universe" -- distinct batch keys plus the
// oldest live ring records, as list nodes in shared memory -- lets one thread replay the exact
// linked-list algorithm over it (refilling candidates on demand), and then all threads apply the
// net effect to HBM in parallel.
#include <algorithm>
#include <vector>

#include <cub/block/block_scan.cuh>

#include "ffc_common.cuh"
#include "identify_internal.cuh"

namespace ffc {

constexpr int NB = FFC_LRU_MAX_BATCH;  // positions per batch
constexpr int NT = 1024;               // threads of the resolve CTA
constexpr int NN = 2 * NB;             // max local nodes
constexpr int LHSZ = 4096;             // local (smem) hash cells
constexpr int HS = NN, TS = NN + 1;    // list sentinels: head (MRU side), tail (LRU side)

enum : uint8_t { F_RES = 1, F_RES0 = 2, F_INLIST = 4, F_TOUCHED = 8 };
enum : uint8_t { K_HIT = 0, K_FRESH = 1, K_EVICT = 2 };

struct LruState {  // device scalars
  int32_t cur_idx;
  int32_t err;
  int64_t head;
  int64_t tail;
  int64_t jlen;
};

struct JournalEntry {
  int64_t new_key;
  int64_t old_key;
  int64_t old_pos;
  int64_t pos;        // ring position of this access (== head before it)
  int64_t tail_before;
  int32_t slot;
  int32_t cur_before;
  uint8_t kind;
  uint8_t old_qpos;
  uint8_t pad[6];
};

}  // namespace ffc

struct ffc_lru {
  int64_t cap, T, RC, jcap;
  int64_t* ht_key;
  int32_t* ht_slot;
  int64_t* slot_key;
  int64_t* last_pos;
  int32_t* ring[2];
  int cur_ring;
  ffc::LruState* st;
  ffc::JournalEntry* journal;
  int32_t* s0;           // [NB] lookup scratch
  int32_t* blk_counts;   // compaction scratch
  int64_t n_blk;
  // conservative host-side counters (no device sync needed to decide on maintenance)
  int64_t ring_used_ub, ht_used_ub, jlen_host;
};

namespace ffc {

// ------------------------------------------------------------------------------------------------
// warp-cooperative hash table primitives (all 32 lanes call with the same key)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int32_t ht_find_warp(const int64_t* __restrict__ ht_key, const int32_t* __restrict__ ht_slot,
                                                int64_t nwin, int64_t key, int lane, int64_t* cell_out) {
  int64_t w = (int64_t)(mix64((uint64_t)key) & (uint64_t)(nwin - 1));
  for (int64_t it = 0; it < nwin; ++it) {
    const int64_t cell = w * 32 + lane;
    const int64_t k = __ldcg(ht_key + cell);
    const unsigned m = __ballot_sync(0xffffffffu, k == key);
    if (m) {
      const int64_t c = w * 32 + (__ffs(m) - 1);
      if (cell_out) *cell_out = c;
      return __ldcg(ht_slot + c);
    }
    if (__ballot_sync(0xffffffffu, k == KEY_EMPTY)) return -1;
    w = (w + 1) & (nwin - 1);
  }
  return -1;
}

__device__ __forceinline__ void ht_delete_warp(int64_t* ht_key, const int32_t* ht_slot, int64_t nwin, int64_t key, int lane) {
  int64_t cell = -1;
  const int32_t s = ht_find_warp(ht_key, ht_slot, nwin, key, lane, &cell);
  if (s >= 0 && lane == 0) ht_key[cell] = KEY_TOMB;
  __syncwarp();
}

// insert a key known to be absent
__device__ __forceinline__ void ht_insert_warp(int64_t* ht_key, int32_t* ht_slot, int64_t nwin, int64_t key, int32_t slot, int lane) {
  int64_t w = (int64_t)(mix64((uint64_t)key) & (uint64_t)(nwin - 1));
  for (int64_t it = 0; it < 4 * nwin; ++it) {
    const int64_t cell = w * 32 + lane;
    const int64_t k = __ldcg(ht_key + cell);
    const unsigned freem = __ballot_sync(0xffffffffu, k == KEY_EMPTY || k == KEY_TOMB);
    if (freem) {
      const int src = __ffs(freem) - 1;
      int ok = 0;
      if (lane == src) {
        const unsigned long long old = atomicCAS((unsigned long long*)(ht_key + cell), (unsigned long long)k, (unsigned long long)key);
        ok = (old == (unsigned long long)k);
        if (ok) ht_slot[cell] = slot;
      }
      ok = __shfl_sync(0xffffffffu, ok, src);
      if (ok) return;
      continue;  // lost the race for that cell: re-read the same window
    }
    w = (w + 1) & (nwin - 1);
  }
}

__device__ __forceinline__ void ht_put_warp(int64_t* ht_key, int32_t* ht_slot, int64_t nwin, int64_t key, int32_t slot, int lane) {
  int64_t cell = -1;
  const int32_t s = ht_find_warp(ht_key, ht_slot, nwin, key, lane, &cell);
  if (s >= 0) {
    if (lane == 0 && s != slot) ht_slot[cell] = slot;
    __syncwarp();
    return;
  }
  ht_insert_warp(ht_key, ht_slot, nwin, key, slot, lane);
}

// ------------------------------------------------------------------------------------------------
// lookup: one warp per key (lru.py:145-151 view / __contains__)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) lru_lookup_kernel(const int64_t* __restrict__ ht_key, const int32_t* __restrict__ ht_slot,
                                                         int64_t nwin, const int64_t* __restrict__ keys, int n,
                                                         int32_t* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (wid >= n) return;
  const int64_t key = keys[wid];
  const int32_t s = ht_find_warp(ht_key, ht_slot, nwin, key, lane, nullptr);
  if (lane == 0) out[wid] = s;
}

// ------------------------------------------------------------------------------------------------
// resolve: one CTA replays the batch
// ------------------------------------------------------------------------------------------------
struct ResolveSmem {
  int32_t ones0, ones1;     // n_ones before / after this launch (R6)
  int32_t ones_pad[2];
  int64_t pkey[NB];
  int64_t nkey[NN];
  int64_t npos[NN];
  int64_t j_oldkey[NB];
  int64_t j_oldpos[NB];
  int32_t nslot[NN];
  int32_t nslot0[NN];
  int32_t lh[LHSZ];
  int32_t firstocc[LHSZ];
  int32_t pcol[NB];
  int32_t j_cur[NB];
  uint16_t pnode[NB];
  uint16_t tmp[NT];
  uint16_t prev[NN + 2];
  uint16_t next[NN + 2];
  uint8_t nflags[NN];
  uint8_t nqpos[NN];
  uint8_t prow[NB];
  uint8_t pkind[NB];
  uint8_t j_oldq[NB];
  uint8_t freshq[NB];
  // control block
  int64_t scan_pos;
  int32_t n_nodes;
  int32_t n_untouched;
  int32_t zf;
  int32_t sim_i;
  int32_t sim_done;
  int32_t want;
  int32_t cur;
  int32_t err;
  typename cub::BlockScan<int, NT>::TempStorage scan;
};

struct ResolveArgs {
  int64_t* ht_key;
  int32_t* ht_slot;
  int64_t nwin;
  int64_t* slot_key;
  int64_t* last_pos;
  int32_t* ring;
  int64_t rmask;
  int64_t cap;
  LruState* st;
  JournalEntry* journal;
  int64_t jcap;
  const int64_t* keys;
  int32_t* s0;          // [NB] table lookups of the current chunk (chunk 0: lru_lookup_kernel; later chunks: the CTA itself)
  int n;
  const int32_t* n_dev;   // optional device-side key count (sharded callers): n_eff = clamp(*n_dev - n_base, 0, n)
  int n_base;
  int do_journal;
  uint8_t* qpos;
  int32_t* rows_out;
  int32_t* cols_out;
  uint8_t* hit_out;
  int32_t* ones_list;
  int32_t* n_ones;
  uint32_t* cmask;
};

__device__ __forceinline__ int lh_find(const ResolveSmem& S, int64_t key) {
  int c = (int)(mix64((uint64_t)key) & (LHSZ - 1));
  while (true) {
    const int cur = S.lh[c];
    if (cur < 0) return -1;
    if (S.pkey[cur] == key) return (int)S.pnode[S.firstocc[c]];
    c = (c + 1) & (LHSZ - 1);
  }
}

// All threads: pull up to `want` more untouched candidates (oldest live ring records) into the list.
__device__ void fetch_candidates(ResolveSmem& S, const ResolveArgs& a, int64_t head, int want) {
  const int tid = threadIdx.x;
  while (true) {
    __syncthreads();
    const int64_t sp = S.scan_pos;
    const int have = S.n_untouched;
    const int base_nodes = S.n_nodes;
    const int zf = S.zf;
    if (have >= want || sp >= head) break;
    const int room = want - have;
    const int64_t pos = sp + tid;
    bool valid = false;
    int32_t slot = -1;
    int64_t key = 0;
    int node = -1;
    if (pos < head) {
      slot = a.ring[pos & a.rmask];
      valid = (__ldcg(a.last_pos + slot) == pos);
      if (valid) {
        key = __ldcg(a.slot_key + slot);
        node = lh_find(S, key);
        if (node >= 0 && (S.nflags[node] & F_TOUCHED)) valid = false;  // already moved to the front in this batch
      }
    }
    int rank, total;
    cub::BlockScan<int, NT>(S.scan).ExclusiveSum(valid ? 1 : 0, rank, total);
    __syncthreads();
    const int take = total < room ? total : room;
    const bool mine = valid && rank < take;
    int nrank, ntotal;
    cub::BlockScan<int, NT>(S.scan).ExclusiveSum((mine && node < 0) ? 1 : 0, nrank, ntotal);
    if (mine) {
      if (node < 0) {
        node = base_nodes + nrank;
        S.nkey[node] = key;
        S.nslot[node] = slot;
        S.nslot0[node] = slot;
        S.nqpos[node] = a.qpos ? a.qpos[slot] : 0;
        S.nflags[node] = F_RES | F_RES0 | F_INLIST;
      } else {
        S.nflags[node] |= F_INLIST;
      }
      S.npos[node] = pos;
      S.tmp[rank] = (uint16_t)node;
    }
    if (valid && rank == take) S.scan_pos = pos;  // first live record NOT taken: rescan from here next time
    __syncthreads();
    if (mine) {
      // chain (MRU side) prev[zf] -> c[take-1] -> ... -> c[0] -> zf (LRU side)
      S.next[node] = (rank == 0) ? (uint16_t)zf : S.tmp[rank - 1];
      S.prev[node] = (rank == take - 1) ? S.prev[zf] : S.tmp[rank + 1];
    }
    __syncthreads();
    if (tid == 0) {
      if (take > 0) {
        const int newest = S.tmp[take - 1], oldest = S.tmp[0];
        const int P = S.prev[newest];
        S.next[P] = (uint16_t)newest;
        S.prev[zf] = (uint16_t)oldest;
        S.zf = newest;
      }
      S.n_untouched = have + take;
      S.n_nodes = base_nodes + ntotal;
      if (take == total) S.scan_pos = sp + NT;
    }
  }
  __syncthreads();
}

__device__ __forceinline__ void list_unlink(ResolveSmem& S, int nd) {
  const int p = S.prev[nd], n = S.next[nd];
  S.next[p] = (uint16_t)n;
  S.prev[n] = (uint16_t)p;
}
__device__ __forceinline__ void list_push_front(ResolveSmem& S, int nd) {
  const int f = S.next[HS];
  S.prev[nd] = HS;
  S.next[nd] = (uint16_t)f;
  S.prev[f] = (uint16_t)nd;
  S.next[HS] = (uint16_t)nd;
}

// thread 0: replay lru.py get()/try_get() + ffc.py:166-177 over the local universe
__device__ void run_sim(ResolveSmem& S, const ResolveArgs& a, int64_t head, int cur0) {
  int cur = S.cur;
  int zf = S.zf;
  int n_unt = S.n_untouched;
  const bool exhausted = S.scan_pos >= head;
  int i = S.sim_i;
  for (; i < a.n; ++i) {
    const int nd = S.pnode[i];
    const uint8_t f = S.nflags[nd];
    int32_t slot;
    uint8_t kind;
    S.j_cur[i] = cur;
    if (f & F_RES) {
      slot = S.nslot[nd];
      kind = K_HIT;
      S.j_oldkey[i] = S.nkey[nd];
      S.j_oldpos[i] = S.npos[nd];
      const uint8_t q = S.nqpos[nd];
      S.j_oldq[i] = q;
      S.prow[i] = q;
      S.nqpos[nd] = q ^ 1;
      if (f & F_INLIST) {
        if (!(f & F_TOUCHED)) {
          --n_unt;
          if (nd == zf) zf = S.next[nd];
        }
        list_unlink(S, nd);
      }
      list_push_front(S, nd);
      S.nflags[nd] = f | F_INLIST | F_TOUCHED;
    } else {
      if (cur < a.cap) {
        slot = cur;
        kind = K_FRESH;
        S.j_oldkey[i] = KEY_EMPTY;
        S.j_oldpos[i] = -1;
        S.j_oldq[i] = S.freshq[cur - cur0];
        ++cur;
      } else {
        if (n_unt == 0 && !exhausted) {  // need older residents that are not local yet
          int w = a.n - i;
          S.want = w < 32 ? w : 32;
          break;
        }
        const int v = S.prev[TS];
        if (v == HS) {  // capacity 0 or corrupted state
          S.err = 3;
          i = a.n;
          break;
        }
        const uint8_t fv = S.nflags[v];
        if (!(fv & F_TOUCHED)) {
          --n_unt;
          if (v == zf) zf = TS;
        }
        list_unlink(S, v);
        S.nflags[v] = fv & ~(F_RES | F_INLIST);
        slot = S.nslot[v];
        kind = K_EVICT;
        S.j_oldkey[i] = S.nkey[v];
        S.j_oldpos[i] = S.npos[v];
        S.j_oldq[i] = S.nqpos[v];
      }
      S.nslot[nd] = slot;
      S.nqpos[nd] = 1;
      S.prow[i] = 0;
      list_push_front(S, nd);
      S.nflags[nd] = (f & ~F_INLIST) | F_RES | F_INLIST | F_TOUCHED;
    }
    S.npos[nd] = head + i;
    S.pcol[i] = slot;
    S.pkind[i] = kind;
  }
  S.cur = cur;
  S.zf = zf;
  S.n_untouched = n_unt;
  S.sim_i = i;
  S.sim_done = (i >= a.n);
}

// One chunk (<= NB keys) of a batch, all threads of the single resolve CTA.  Returns false when the device error flag was raised.
__device__ bool resolve_chunk(const ResolveArgs& a, ResolveSmem& S) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = a.n;
  LruState* st = a.st;
  const int cur0 = st->cur_idx;
  const int64_t head = st->head, tail = st->tail, jlen = st->jlen;

  // ring / journal capacity guards (host keeps conservative counters; this is the backstop)
  if (head + n - tail > a.rmask + 1 || (a.do_journal && jlen + n > a.jcap)) {
    if (tid == 0) st->err = (head + n - tail > a.rmask + 1) ? 1 : 2;
    return false;
  }

  for (int c = tid; c < LHSZ; c += NT) {
    S.lh[c] = -1;
    S.firstocc[c] = 0x7fffffff;
  }
  if (tid == 0 && a.ones_list) S.ones0 = *reinterpret_cast<volatile int32_t*>(a.n_ones);
  int64_t key = 0;
  int32_t s0 = -1;
  if (tid < n) {
    key = a.keys[tid];
    s0 = a.s0[tid];
    S.pkey[tid] = key;
    const int fs = cur0 + tid;
    S.freshq[tid] = (a.qpos && fs < a.cap) ? a.qpos[fs] : 0;
  }
  if (tid == 0) {
    S.next[HS] = TS;
    S.prev[TS] = HS;
    S.prev[HS] = HS;
    S.next[TS] = TS;
    S.scan_pos = tail;
    S.n_untouched = 0;
    S.zf = TS;
    S.sim_i = 0;
    S.sim_done = 0;
    S.want = 0;
    S.cur = cur0;
    S.err = 0;
  }
  __syncthreads();

  // R1: dedupe batch keys -> first occurrence -> node ids
  int mycell = -1;
  if (tid < n) {
    int c = (int)(mix64((uint64_t)key) & (LHSZ - 1));
    while (true) {
      int curp = S.lh[c];
      if (curp < 0) {
        const int old = atomicCAS(&S.lh[c], -1, tid);
        if (old < 0) break;
        curp = old;
      }
      if (S.pkey[curp] == key) break;
      c = (c + 1) & (LHSZ - 1);
    }
    mycell = c;
    atomicMin(&S.firstocc[c], tid);
  }
  __syncthreads();
  const bool is_first = (tid < n) && (S.firstocc[mycell] == tid);
  int nid, n_distinct;
  cub::BlockScan<int, NT>(S.scan).ExclusiveSum(is_first ? 1 : 0, nid, n_distinct);
  if (is_first) {
    S.pnode[tid] = (uint16_t)nid;
    S.nkey[nid] = key;
    S.nslot[nid] = s0;
    S.nslot0[nid] = s0;
    S.nflags[nid] = (s0 >= 0) ? (F_RES | F_RES0) : 0;
    S.npos[nid] = (s0 >= 0) ? __ldcg(a.last_pos + s0) : -1;
    S.nqpos[nid] = (s0 >= 0 && a.qpos) ? a.qpos[s0] : 0;
  }
  const int n_miss0 = __syncthreads_count(is_first && s0 < 0);
  if (tid < n && !is_first) S.pnode[tid] = S.pnode[S.firstocc[mycell]];
  if (tid == 0) S.n_nodes = n_distinct;
  __syncthreads();

  const int64_t fresh_room = a.cap - cur0;
  if ((int64_t)n_miss0 <= fresh_room) {
    // ---- fast path: no eviction can happen (all hits and/or fresh slots) => every position resolves independently:
    // a key's j-th occurrence in the batch is a hit except a new key's first one; rows follow the qpos parity;
    // the m-th new key (in batch order) takes slot cur_idx + m.  (lru.py:44-89 + ffc.py:166-177, closed form)
    int* cnt = S.lh;              // [n_nodes] occurrences per node   (the smem hash is not needed any more)
    int* lastp = S.lh + NB;       // [n_nodes] last position per node
    __syncthreads();
    for (int c = tid; c < 2 * NB; c += NT) S.lh[c] = 0;
    __syncthreads();
    int nd = 0, occ = 0, prevpos = -1;
    if (tid < n) {
      nd = S.pnode[tid];
      for (int j = 0; j < tid; ++j)
        if (S.pnode[j] == nd) {
          ++occ;
          prevpos = j;
        }
      atomicAdd(&cnt[nd], 1);
      atomicMax(&lastp[nd], tid);
    }
    const bool fresh_here = (tid < n) && occ == 0 && !(S.nflags[nd] & F_RES0);
    int frank, ftotal;
    cub::BlockScan<int, NT>(S.scan).ExclusiveSum(fresh_here ? 1 : 0, frank, ftotal);
    if (fresh_here) S.nslot[nd] = cur0 + frank;
    __syncthreads();
    if (tid < n) {
      const bool res0 = S.nflags[nd] & F_RES0;
      const int32_t slot = S.nslot[nd];
      uint8_t row, kind, oldq;
      int64_t oldkey, oldpos;
      if (res0) {
        kind = K_HIT;
        row = S.nqpos[nd] ^ (uint8_t)(occ & 1);
        oldq = row;
        oldkey = key;
        oldpos = occ == 0 ? S.npos[nd] : head + prevpos;
      } else if (occ == 0) {
        kind = K_FRESH;
        row = 0;
        oldq = S.freshq[slot - cur0];
        oldkey = KEY_EMPTY;
        oldpos = -1;
      } else {
        kind = K_HIT;
        row = 1 ^ (uint8_t)((occ - 1) & 1);
        oldq = row;
        oldkey = key;
        oldpos = head + prevpos;
      }
      S.pcol[tid] = slot;
      S.prow[tid] = row;
      S.pkind[tid] = kind;
      S.j_oldkey[tid] = oldkey;
      S.j_oldpos[tid] = oldpos;
      S.j_oldq[tid] = oldq;
      S.j_cur[tid] = cur0 + frank;
    }
    __syncthreads();
    if (tid < n && lastp[nd] == tid) {   // the last occurrence finalises the node
      const bool res0 = S.nflags[nd] & F_RES0;
      const int c = cnt[nd];
      S.nqpos[nd] = res0 ? (S.nqpos[nd] ^ (uint8_t)(c & 1)) : (uint8_t)(1 ^ ((c - 1) & 1));
      S.npos[nd] = head + tid;
      S.nflags[nd] |= F_RES | F_TOUCHED;
    }
    if (tid == 0) S.cur = cur0 + ftotal;
    __syncthreads();
  } else {
    // R2: initial candidates = number of evictions the batch needs if no resident entry is endangered
    {
      int64_t need = (int64_t)n_miss0 - fresh_room;
      if (need > 0) fetch_candidates(S, a, head, (int)need);
    }
    // R3: sequential replay with on-demand refill
    while (true) {
      if (tid == 0) run_sim(S, a, head, cur0);
      __syncthreads();
      if (S.sim_done) break;
      const int want = S.want;
      fetch_candidates(S, a, head, want);
      if (tid == 0 && S.n_untouched == 0 && S.scan_pos < head) S.err = 4;  // cannot happen
    }
  }
  if (S.err) {
    if (tid == 0) st->err = S.err;
    return false;
  }

  // R4: outputs
  if (tid < n) {
    const int32_t slot = S.pcol[tid];
    const uint8_t kind = S.pkind[tid];
    a.cols_out[tid] = slot;
    if (a.rows_out) a.rows_out[tid] = S.prow[tid];
    if (a.hit_out) a.hit_out[tid] = (kind == K_HIT);
    if (kind == K_HIT && a.cmask) {
      const uint32_t bit = 1u << (slot & 31);
      const uint32_t old = atomicOr(a.cmask + (slot >> 5), bit);
      if (!(old & bit) && a.ones_list) {
        const int idx = atomicAdd(a.n_ones, 1);
        a.ones_list[idx] = slot;
      }
    }
    a.ring[(head + tid) & a.rmask] = slot;
    if (a.do_journal) {
      JournalEntry e;
      e.new_key = key;
      e.old_key = S.j_oldkey[tid];
      e.old_pos = S.j_oldpos[tid];
      e.pos = head + tid;
      e.tail_before = tail;
      e.slot = slot;
      e.cur_before = S.j_cur[tid];
      e.kind = kind;
      e.old_qpos = S.j_oldq[tid];
      for (int b = 0; b < 6; ++b) e.pad[b] = 0;
      a.journal[jlen + tid] = e;
    }
  }
  // R5: net effect on per-slot state, then hash table (deletes before inserts)
  const int n_nodes = S.n_nodes;
  for (int t = tid; t < n_nodes; t += NT) {
    const uint8_t f = S.nflags[t];
    if ((f & F_RES) && (f & F_TOUCHED)) {
      const int32_t slot = S.nslot[t];
      a.slot_key[slot] = S.nkey[t];
      a.last_pos[slot] = S.npos[t];
      if (a.qpos) a.qpos[slot] = S.nqpos[t];
    }
  }
  for (int t = warp; t < n_nodes; t += NT / 32) {
    const uint8_t f = S.nflags[t];
    const bool res = f & F_RES, res0 = f & F_RES0;
    if (res0 && (!res || S.nslot[t] != S.nslot0[t])) ht_delete_warp(a.ht_key, a.ht_slot, a.nwin, S.nkey[t], lane);
  }
  __syncthreads();
  for (int t = warp; t < n_nodes; t += NT / 32) {
    const uint8_t f = S.nflags[t];
    const bool res = f & F_RES, res0 = f & F_RES0;
    if (res && (!res0 || S.nslot[t] != S.nslot0[t])) ht_insert_warp(a.ht_key, a.ht_slot, a.nwin, S.nkey[t], S.nslot[t], lane);
  }
  if (tid == 0) {
    st->cur_idx = S.cur;
    st->head = head + n;
    if (a.do_journal) {
      st->jlen = jlen + n;
    } else {
      // everything before the oldest untouched local candidate (or the scan position) is dead now
      const int last = S.prev[TS];
      int64_t nt = S.scan_pos;
      if (last != HS && !(S.nflags[last] & F_TOUCHED)) nt = S.npos[last];
      if (nt > head) nt = head;
      st->tail = nt;
    }
  }
  // R6: `ones` is a set (ffc.py:170/226 ones_idx), but the list is appended with atomics in arrival order; sort this launch's
  // segment by slot so that the list -- and with it the gather / summation order of the side sweeps -- is run-to-run deterministic
  if (a.ones_list) {
    __syncthreads();                              // all R4 appends of this (single) CTA are done
    if (tid == 0) S.ones1 = *reinterpret_cast<volatile int32_t*>(a.n_ones);
    __syncthreads();
    const int n0 = S.ones0, len = S.ones1 - n0;   // len <= n <= NT
    int32_t mine = 0;
    if (tid < len) {
      mine = *reinterpret_cast<volatile int32_t*>(a.ones_list + n0 + tid);
      S.lh[tid] = mine;                           // the local hash is dead by now: scratch
    }
    __syncthreads();
    if (tid < len) {
      int rank = 0;
      for (int j = 0; j < len; ++j) rank += S.lh[j] < mine ? 1 : 0;     // slots are distinct
      a.ones_list[n0 + rank] = mine;
    }
  }
  return true;
}

// ONE launch per batch of any size: the CTA walks the batch in chunks of NB keys (the reference semantics are sequential, so
// chunks cannot run side by side).  The table lookups of chunk 0 come from lru_lookup_kernel (many CTAs, launched just before);
// later chunks depend on the inserts / evictions of the earlier ones, so the CTA looks their keys up itself (one warp per key).
// With a device-side key count (sharded callers) the walk stops at clamp(*n_dev - n_base, 0, n): no empty launches.
__global__ void __launch_bounds__(NT, 1) lru_resolve_kernel(const ResolveArgs a_in) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ResolveSmem& S = *reinterpret_cast<ResolveSmem*>(smem_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int n_total = a_in.n;
  if (a_in.n_dev) {
    n_total = *a_in.n_dev - a_in.n_base;
    n_total = n_total < 0 ? 0 : (n_total > a_in.n ? a_in.n : n_total);
  }
  for (int base = 0; base < n_total; base += NB) {
    ResolveArgs a = a_in;
    a.n = n_total - base < NB ? n_total - base : NB;
    a.keys += base;
    a.cols_out += base;
    if (a.rows_out) a.rows_out += base;
    if (a.hit_out) a.hit_out += base;
    if (base > 0) {
      __syncthreads();      // the previous chunk's table / state updates are complete
      for (int t = warp; t < a.n; t += NT / 32) {
        const int32_t s = ht_find_warp(a.ht_key, a.ht_slot, a.nwin, a.keys[t], lane, nullptr);
        if (lane == 0) a.s0[t] = s;
      }
      __syncthreads();
    }
    if (!resolve_chunk(a, S)) return;
  }
}

// ------------------------------------------------------------------------------------------------
// undo (lru.py:210-255 rollback_steps + ffc.py:256-257 qpos restore)
// ------------------------------------------------------------------------------------------------
struct UndoSmem {
  JournalEntry e[NB];
  int32_t sh[LHSZ];      // slot hash: slot value or -1
  int32_t shmin[LHSZ];   // earliest entry index for that slot
  int32_t shmut[LHSZ];   // 1 if any entry of that slot changed its key (fresh / evict)
};

__global__ void __launch_bounds__(NT, 1) lru_undo_kernel(int64_t* ht_key, int32_t* ht_slot, int64_t nwin, int64_t* slot_key,
                                                          int64_t* last_pos, LruState* st, const JournalEntry* journal,
                                                          int64_t steps, uint8_t* qpos) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  UndoSmem& S = *reinterpret_cast<UndoSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t jl = st->jlen;
  const int64_t m = steps < jl ? steps : jl;
  const int64_t lo = jl - m;
  for (int64_t hi = jl; hi > lo;) {
    const int64_t a = (hi - lo > NB) ? hi - NB : lo;
    const int cnt = (int)(hi - a);
    for (int c = tid; c < LHSZ; c += NT) {
      S.sh[c] = -1;
      S.shmin[c] = 0x7fffffff;
      S.shmut[c] = 0;
    }
    if (tid < cnt) S.e[tid] = journal[a + tid];
    __syncthreads();
    int mycell = -1;
    if (tid < cnt) {
      const int32_t slot = S.e[tid].slot;
      int c = (int)(mix64((uint64_t)slot) & (LHSZ - 1));
      while (true) {
        int cur = S.sh[c];
        if (cur < 0) {
          const int old = atomicCAS(&S.sh[c], -1, slot);
          if (old < 0) break;
          cur = old;
        }
        if (cur == slot) break;
        c = (c + 1) & (LHSZ - 1);
      }
      mycell = c;
      atomicMin(&S.shmin[c], tid);
      if (S.e[tid].kind != K_HIT) S.shmut[c] = 1;
    }
    __syncthreads();
    // phase 1: remove every key this range inserted
    for (int t = warp; t < cnt; t += NT / 32) {
      if (S.e[t].kind != K_HIT) ht_delete_warp(ht_key, ht_slot, nwin, S.e[t].new_key, lane);
    }
    __syncthreads();
    // phase 2: the earliest entry of each slot restores the slot and its old key's mapping
    if (tid < cnt && S.shmin[mycell] == tid) {
      const JournalEntry& e = S.e[tid];
      slot_key[e.slot] = e.old_key;
      last_pos[e.slot] = e.old_pos;
      if (qpos) qpos[e.slot] = e.old_qpos;
    }
    for (int t = warp; t < cnt; t += NT / 32) {
      const JournalEntry& e = S.e[t];
      int c = (int)(mix64((uint64_t)e.slot) & (LHSZ - 1));
      while (S.sh[c] != e.slot) c = (c + 1) & (LHSZ - 1);
      // a slot that only saw hits still maps its key: nothing to repair in the table
      if (S.shmin[c] == t && e.kind != K_FRESH && S.shmut[c]) ht_put_warp(ht_key, ht_slot, nwin, e.old_key, e.slot, lane);
    }
    __syncthreads();
    if (tid == 0) {
      st->cur_idx = S.e[0].cur_before;
      st->head = S.e[0].pos;
      st->tail = S.e[0].tail_before;
    }
    __syncthreads();
    hi = a;
  }
  if (tid == 0) st->jlen = lo;
}

// ------------------------------------------------------------------------------------------------
// maintenance: ring compaction (order-preserving) and hash-table rebuild
// ------------------------------------------------------------------------------------------------
__global__ void fill_i64_kernel(int64_t* p, int64_t n, int64_t v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

__global__ void __launch_bounds__(1024) ring_count_kernel(const int32_t* __restrict__ ring, int64_t rmask, const int64_t* __restrict__ last_pos,
                                                          const LruState* st, int32_t* blk_counts) {
  const int64_t tail = st->tail, head = st->head;
  const int64_t pos = tail + (int64_t)blockIdx.x * 1024 + threadIdx.x;
  bool valid = false;
  if (pos < head) {
    const int32_t slot = ring[pos & rmask];
    valid = (last_pos[slot] == pos);
  }
  const int c = __syncthreads_count(valid);
  if (threadIdx.x == 0) blk_counts[blockIdx.x] = c;
}

__global__ void __launch_bounds__(1024) ring_scan_kernel(int32_t* blk_counts, int64_t n_blk, int64_t* total_out) {
  // single block exclusive scan over n_blk counts (n_blk <= a few thousand)
  __shared__ typename cub::BlockScan<int, 1024>::TempStorage tmp;
  int carry = 0;
  for (int64_t base = 0; base < n_blk; base += 1024) {
    const int64_t i = base + threadIdx.x;
    const int v = (i < n_blk) ? blk_counts[i] : 0;
    int ex, tot;
    cub::BlockScan<int, 1024>(tmp).ExclusiveSum(v, ex, tot);
    if (i < n_blk) blk_counts[i] = carry + ex;
    carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(1024) ring_move_kernel(const int32_t* __restrict__ ring_old, int32_t* __restrict__ ring_new, int64_t rmask,
                                                         int64_t* last_pos, const LruState* st, const int32_t* blk_offsets) {
  __shared__ typename cub::BlockScan<int, 1024>::TempStorage tmp;
  const int64_t tail = st->tail, head = st->head;
  const int64_t pos = tail + (int64_t)blockIdx.x * 1024 + threadIdx.x;
  bool valid = false;
  int32_t slot = -1;
  if (pos < head) {
    slot = ring_old[pos & rmask];
    valid = (last_pos[slot] == pos);
  }
  int ex;
  cub::BlockScan<int, 1024>(tmp).ExclusiveSum(valid ? 1 : 0, ex);
  if (valid) {
    const int64_t np = head + blk_offsets[blockIdx.x] + ex;
    ring_new[np & rmask] = slot;
    last_pos[slot] = np;
  }
}

__global__ void ring_commit_kernel(LruState* st, const int64_t* total) {
  const int64_t head = st->head;
  st->tail = head;
  st->head = head + *total;
}

__global__ void __launch_bounds__(256) ht_rebuild_kernel(int64_t* ht_key, int32_t* ht_slot, int64_t nwin, const int64_t* __restrict__ slot_key,
                                                         const LruState* st) {
  const int lane = threadIdx.x & 31;
  const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int cur = st->cur_idx;
  for (int64_t s = wid; s < cur; s += nw) {
    const int64_t key = slot_key[s];
    if (key != KEY_EMPTY) ht_insert_warp(ht_key, ht_slot, nwin, key, (int32_t)s, lane);
  }
}

__global__ void lru_reset_state_kernel(LruState* st) {
  st->cur_idx = 0;
  st->err = 0;
  st->head = 0;
  st->tail = 0;
  st->jlen = 0;
}

static int lru_fill(int64_t* p, int64_t n, int64_t v, cudaStream_t s) {
  int blocks = (int)std::min<int64_t>(ceil_div64(n, 256), 148 * 8);
  if (blocks < 1) blocks = 1;
  fill_i64_kernel<<<blocks, 256, 0, s>>>(p, n, v);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

static int lru_rebuild_ht(ffc_lru* h, cudaStream_t s) {
  int rc = lru_fill(h->ht_key, h->T, KEY_EMPTY, s);
  if (rc) return rc;
  ht_rebuild_kernel<<<148 * 4, 256, 0, s>>>(h->ht_key, h->ht_slot, h->T / 32, h->slot_key, h->st);
  FFC_LAUNCH_CHECK();
  h->ht_used_ub = h->cap;
  return FFC_OK;
}

static int lru_compact_ring(ffc_lru* h, cudaStream_t s) {
  // the live span is at most ring_used_ub records long
  const int64_t span = std::min<int64_t>(h->ring_used_ub, h->RC);
  const int64_t n_blk = std::max<int64_t>(1, ceil_div64(span, 1024));
  if (n_blk > h->n_blk) {
    set_error("ring compaction scratch too small");
    return FFC_ERR_STATE;
  }
  int32_t* oldr = h->ring[h->cur_ring];
  int32_t* newr = h->ring[h->cur_ring ^ 1];
  int64_t* total = reinterpret_cast<int64_t*>(h->blk_counts + h->n_blk);
  ring_count_kernel<<<(int)n_blk, 1024, 0, s>>>(oldr, h->RC - 1, h->last_pos, h->st, h->blk_counts);
  FFC_LAUNCH_CHECK();
  ring_scan_kernel<<<1, 1024, 0, s>>>(h->blk_counts, n_blk, total);
  FFC_LAUNCH_CHECK();
  ring_move_kernel<<<(int)n_blk, 1024, 0, s>>>(oldr, newr, h->RC - 1, h->last_pos, h->st, h->blk_counts);
  FFC_LAUNCH_CHECK();
  ring_commit_kernel<<<1, 1, 0, s>>>(h->st, total);
  FFC_LAUNCH_CHECK();
  h->cur_ring ^= 1;
  h->ring_used_ub = h->cap;
  return FFC_OK;
}

static int lru_check_err(ffc_lru* h, cudaStream_t s) {
  int32_t err = 0;
  FFC_CUDA(cudaMemcpyAsync(&err, &h->st->err, sizeof(err), cudaMemcpyDeviceToHost, s));
  FFC_CUDA(cudaStreamSynchronize(s));
  if (err) {
    set_error("device LRU error flag %d (1=ring full, 2=journal full, 3=empty cache with zero capacity, 4=scan)", err);
    return FFC_ERR_STATE;
  }
  return FFC_OK;
}

}  // namespace ffc

using namespace ffc;

extern "C" int ffc_lru_create(int64_t capacity, int64_t journal_capacity, ffc_lru_t** out) {
  FFC_REQUIRE(out != nullptr, "ffc_lru_create: out is NULL");
  FFC_REQUIRE(capacity >= 1 && capacity <= (int64_t)1 << 30, "ffc_lru_create: capacity %lld out of range", (long long)capacity);
  ffc_lru* h = new ffc_lru();
  memset(h, 0, sizeof(*h));
  h->cap = capacity;
  // 4x the capacity, and never less than 2^18: one pass may bring FFC_LRU_MAX_KEYS accesses (plus as many journaled ones
  // outstanding) on top of `capacity` live records, whatever the capacity
  h->T = std::max<int64_t>(next_pow2(4 * capacity), (int64_t)1 << 18);
  h->RC = std::max<int64_t>(next_pow2(4 * capacity), (int64_t)1 << 18);
  h->jcap = journal_capacity > 0 ? journal_capacity : 65536;
  h->n_blk = ceil_div64(h->RC, 1024);
  FFC_CUDA(cudaMalloc(&h->ht_key, h->T * sizeof(int64_t)));
  FFC_CUDA(cudaMalloc(&h->ht_slot, h->T * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->slot_key, capacity * sizeof(int64_t)));
  FFC_CUDA(cudaMalloc(&h->last_pos, capacity * sizeof(int64_t)));
  FFC_CUDA(cudaMalloc(&h->ring[0], h->RC * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->ring[1], h->RC * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->st, sizeof(LruState)));
  FFC_CUDA(cudaMalloc(&h->journal, h->jcap * sizeof(JournalEntry)));
  FFC_CUDA(cudaMalloc(&h->s0, NB * sizeof(int32_t)));
  FFC_CUDA(cudaMalloc(&h->blk_counts, h->n_blk * sizeof(int32_t) + 16));
  FFC_CUDA(cudaFuncSetAttribute(lru_resolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ResolveSmem)));
  FFC_CUDA(cudaFuncSetAttribute(lru_undo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(UndoSmem)));
  int rc = ffc_lru_clear(h, nullptr);
  if (rc) return rc;
  FFC_CUDA(cudaStreamSynchronize(nullptr));
  *out = h;
  return FFC_OK;
}

extern "C" int ffc_lru_destroy(ffc_lru_t* h) {
  if (!h) return FFC_OK;
  cudaFree(h->ht_key);
  cudaFree(h->ht_slot);
  cudaFree(h->slot_key);
  cudaFree(h->last_pos);
  cudaFree(h->ring[0]);
  cudaFree(h->ring[1]);
  cudaFree(h->st);
  cudaFree(h->journal);
  cudaFree(h->s0);
  cudaFree(h->blk_counts);
  delete h;
  return FFC_OK;
}

extern "C" int ffc_lru_clear(ffc_lru_t* h, void* stream) {
  FFC_REQUIRE(h != nullptr, "ffc_lru_clear: NULL handle");
  cudaStream_t s = (cudaStream_t)stream;
  int rc;
  if ((rc = lru_fill(h->ht_key, h->T, KEY_EMPTY, s))) return rc;
  if ((rc = lru_fill(h->slot_key, h->cap, KEY_EMPTY, s))) return rc;
  if ((rc = lru_fill(h->last_pos, h->cap, -1, s))) return rc;
  lru_reset_state_kernel<<<1, 1, 0, s>>>(h->st);
  FFC_LAUNCH_CHECK();
  h->cur_ring = 0;
  h->ring_used_ub = 0;
  h->ht_used_ub = 0;
  h->jlen_host = 0;
  return FFC_OK;
}

// Make room for `reserve` more accesses (the WHOLE batch about to be resolved, not one chunk of it: once its first journaled
// chunk is outstanding nothing can be compacted any more).
static int lru_maintain_for(ffc_lru_t* h, int64_t reserve, cudaStream_t s) {
  int rc = FFC_OK;
  if (h->jlen_host == 0 && h->ring_used_ub + reserve + 2 * NB > h->RC) rc = lru_compact_ring(h, s);
  if (rc) return rc;
  if (h->jlen_host == 0 && h->ht_used_ub + 2 * reserve + 2 * NB > h->T / 2) rc = lru_rebuild_ht(h, s);
  return rc;
}

extern "C" int ffc_lru_maintain(ffc_lru_t* h, void* stream) {
  FFC_REQUIRE(h != nullptr, "ffc_lru_maintain: NULL handle");
  return lru_maintain_for(h, 0, (cudaStream_t)stream);
}

extern "C" int ffc_lru_view(ffc_lru_t* h, const int64_t* keys_dev, int n, int32_t* slots_out, void* stream) {
  FFC_REQUIRE(h && keys_dev && slots_out && n >= 1, "ffc_lru_view: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  const int blocks = (int)ceil_div64((int64_t)n * 32, 256);
  lru_lookup_kernel<<<blocks, 256, 0, s>>>(h->ht_key, h->ht_slot, h->T / 32, keys_dev, n, slots_out);
  FFC_LAUNCH_CHECK();
  return FFC_OK;
}

extern "C" int ffc_lru_assign(ffc_lru_t* h, const int64_t* keys_dev, int n, int journal, uint8_t* qpos_dev, int32_t* rows_out,
                              int32_t* cols_out, uint8_t* hit_out, int32_t* ones_list_dev, int32_t* n_ones_dev, uint32_t* cmask_dev,
                              const int32_t* n_dev, int n_base, void* stream) {
  FFC_REQUIRE(h && keys_dev && cols_out, "ffc_lru_assign: NULL argument");
  FFC_REQUIRE(n >= 1 && n <= FFC_LRU_MAX_KEYS, "ffc_lru_assign: n=%d outside [1,%d]", n, FFC_LRU_MAX_KEYS);
  FFC_REQUIRE(!ones_list_dev || (n_ones_dev && cmask_dev), "ffc_lru_assign: ones_list needs n_ones and cmask");
  cudaStream_t s = (cudaStream_t)stream;
  int rc = lru_maintain_for(h, n, s);
  if (rc) return rc;
  if (journal) FFC_REQUIRE(h->jlen_host + n <= h->jcap, "ffc_lru_assign: journal capacity %lld exceeded", (long long)h->jcap);
  if (h->ring_used_ub + n > h->RC) {
    set_error("ffc_lru_assign: recency ring full with %lld journaled accesses outstanding; undo or commit first", (long long)h->jlen_host);
    return FFC_ERR_STATE;
  }
  rc = ffc_lru_view(h, keys_dev, std::min(n, NB), h->s0, s);     // chunk 0; the resolve CTA looks later chunks up itself
  if (rc) return rc;
  ResolveArgs a;
  a.ht_key = h->ht_key;
  a.ht_slot = h->ht_slot;
  a.nwin = h->T / 32;
  a.slot_key = h->slot_key;
  a.last_pos = h->last_pos;
  a.ring = h->ring[h->cur_ring];
  a.rmask = h->RC - 1;
  a.cap = h->cap;
  a.st = h->st;
  a.journal = h->journal;
  a.jcap = h->jcap;
  a.keys = keys_dev;
  a.s0 = h->s0;
  a.n = n;
  a.n_dev = n_dev;
  a.n_base = n_base;
  a.do_journal = journal ? 1 : 0;
  a.qpos = qpos_dev;
  a.rows_out = rows_out;
  a.cols_out = cols_out;
  a.hit_out = hit_out;
  a.ones_list = ones_list_dev;
  a.n_ones = n_ones_dev;
  a.cmask = cmask_dev;
  lru_resolve_kernel<<<1, NT, sizeof(ResolveSmem), s>>>(a);
  FFC_LAUNCH_CHECK();
  h->ring_used_ub += n;
  h->ht_used_ub += n;
  if (journal) h->jlen_host += n;
  return FFC_OK;
}

extern "C" int ffc_lru_undo(ffc_lru_t* h, int64_t steps, uint8_t* qpos_dev, void* stream) {
  FFC_REQUIRE(h != nullptr, "ffc_lru_undo: NULL handle");
  cudaStream_t s = (cudaStream_t)stream;
  if (steps < 0) steps = h->jlen_host;   // everything outstanding (the device-side journal length decides)
  const int64_t m = std::min<int64_t>(steps, h->jlen_host);
  if (m == 0) return FFC_OK;
  lru_undo_kernel<<<1, NT, sizeof(UndoSmem), s>>>(h->ht_key, h->ht_slot, h->T / 32, h->slot_key, h->last_pos, h->st, h->journal, m, qpos_dev);
  FFC_LAUNCH_CHECK();
  h->jlen_host -= m;
  h->ring_used_ub -= m;  // the undone accesses' ring records are gone (head is rolled back)
  h->ht_used_ub += m;    // re-inserted old keys may consume never-used cells
  return FFC_OK;
}

namespace ffc {
int lru_device_state(const ffc_lru_t* h, const int32_t** cur_idx_dev, const int64_t** slot_key, int64_t* capacity) {
  FFC_REQUIRE(h != nullptr, "NULL LRU handle");
  *cur_idx_dev = &h->st->cur_idx;
  *slot_key = h->slot_key;
  *capacity = h->cap;
  return FFC_OK;
}
}  // namespace ffc

extern "C" int ffc_lru_size(ffc_lru_t* h, int64_t* cur_idx_out, int64_t* journal_len_out, void* stream) {
  FFC_REQUIRE(h != nullptr, "ffc_lru_size: NULL handle");
  cudaStream_t s = (cudaStream_t)stream;
  LruState st;
  FFC_CUDA(cudaMemcpyAsync(&st, h->st, sizeof(st), cudaMemcpyDeviceToHost, s));
  FFC_CUDA(cudaStreamSynchronize(s));
  if (st.err) {
    set_error("device LRU error flag %d (1=ring full, 2=journal full, 3=empty cache, 4=scan)", st.err);
    return FFC_ERR_STATE;
  }
  if (cur_idx_out) *cur_idx_out = st.cur_idx;
  if (journal_len_out) *journal_len_out = st.jlen;
  return FFC_OK;
}

extern "C" int ffc_lru_export(ffc_lru_t* h, int64_t* keys_host, int32_t* slots_host, int64_t* n_out, void* stream) {
  FFC_REQUIRE(h && keys_host && slots_host && n_out, "ffc_lru_export: NULL argument");
  cudaStream_t s = (cudaStream_t)stream;
  int rc = lru_check_err(h, s);
  if (rc) return rc;
  LruState st;
  FFC_CUDA(cudaMemcpyAsync(&st, h->st, sizeof(st), cudaMemcpyDeviceToHost, s));
  FFC_CUDA(cudaStreamSynchronize(s));
  const int64_t n = st.cur_idx;
  std::vector<int64_t> keys(n), pos(n);
  if (n > 0) {
    FFC_CUDA(cudaMemcpyAsync(keys.data(), h->slot_key, n * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    FFC_CUDA(cudaMemcpyAsync(pos.data(), h->last_pos, n * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    FFC_CUDA(cudaStreamSynchronize(s));
  }
  std::vector<int32_t> order(n);
  for (int64_t i = 0; i < n; ++i) order[i] = (int32_t)i;
  std::sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return pos[a] > pos[b]; });
  for (int64_t i = 0; i < n; ++i) {
    keys_host[i] = keys[order[i]];
    slots_host[i] = order[i];
  }
  *n_out = n;
  return FFC_OK;
}

namespace ffc {
__global__ void lru_import_state_kernel(LruState* st, int32_t n) {
  st->cur_idx = n;
  st->head = n;
  st->tail = 0;
  st->jlen = 0;
  st->err = 0;
}
}  // namespace ffc

extern "C" int ffc_lru_import(ffc_lru_t* h, const int64_t* keys_host, const int32_t* slots_host, int64_t n, void* stream) {
  FFC_REQUIRE(h && (n == 0 || (keys_host && slots_host)), "ffc_lru_import: NULL argument");
  FFC_REQUIRE(n >= 0 && n <= h->cap, "ffc_lru_import: %lld pairs exceed capacity %lld", (long long)n, (long long)h->cap);
  cudaStream_t s = (cudaStream_t)stream;
  int64_t cur = 0;
  int rc = ffc_lru_size(h, &cur, nullptr, s);
  if (rc) return rc;
  FFC_REQUIRE(cur == 0, "ffc_lru_import: cache not empty (cur_idx=%lld); lru.py:115 asserts cur_idx == 0", (long long)cur);
  std::vector<int64_t> skey(n), spos(n);
  std::vector<int32_t> ring(n);
  std::vector<char> seen(n, 0);
  for (int64_t i = 0; i < n; ++i) {
    const int32_t sl = slots_host[i];
    FFC_REQUIRE(sl >= 0 && sl < n && !seen[sl], "ffc_lru_import: slots must be a permutation of [0,%lld)", (long long)n);
    FFC_REQUIRE(keys_host[i] != KEY_EMPTY && keys_host[i] != KEY_TOMB, "ffc_lru_import: reserved key value");
    seen[sl] = 1;
    skey[sl] = keys_host[i];
    spos[sl] = n - 1 - i;       // pair 0 is the most recent
    ring[n - 1 - i] = sl;
  }
  {
    std::vector<int64_t> sorted(keys_host, keys_host + n);
    std::sort(sorted.begin(), sorted.end());
    FFC_REQUIRE(std::adjacent_find(sorted.begin(), sorted.end()) == sorted.end(), "ffc_lru_import: duplicate key");
  }
  rc = ffc_lru_clear(h, s);
  if (rc) return rc;
  if (n > 0) {
    FFC_CUDA(cudaMemcpyAsync(h->slot_key, skey.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    FFC_CUDA(cudaMemcpyAsync(h->last_pos, spos.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    FFC_CUDA(cudaMemcpyAsync(h->ring[0], ring.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  }
  lru_import_state_kernel<<<1, 1, 0, s>>>(h->st, (int32_t)n);
  FFC_LAUNCH_CHECK();
  rc = lru_rebuild_ht(h, s);
  if (rc) return rc;
  FFC_CUDA(cudaStreamSynchronize(s));  // host vectors go out of scope
  h->ring_used_ub = n;
  return FFC_OK;
}
