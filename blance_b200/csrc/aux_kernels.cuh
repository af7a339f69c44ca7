// blance_b200/csrc/aux_kernels.cuh — the data-parallel kernels around the
// sequential assign pass: row filtering, weighted node histogram, partition sort
// keys, convergence compare/commit, row (un)packing, and CalcPartitionMoves.
// All are one-thread-per-partition, HBM-streaming kernels over the pooled arrays
// (see device_types.cuh); grids are sized as multiples of the SM count by the host.
#pragma once

#include <cuda_runtime.h>

#include "blance_b200.h"
#include "device_types.cuh"

namespace blance_dev {

// ---- H2D side: caller layout -> device layout -----------------------------------------
// rows [PU][SL] -> [PU][SLP] (padded with NO_NODE); shapes uint8[PU][S] -> 2-bit fields.
__global__ void k_unpack(DPool pool, const int32_t* __restrict__ raw_cur, const int32_t* __restrict__ raw_prev,
                         const uint8_t* __restrict__ cur_shape, const uint8_t* __restrict__ prev_shape,
                         const long long* __restrict__ raw_rows_off, const long long* __restrict__ raw_shape_off,
                         long long n_parts_total) {
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n_parts_total;
       g += (long long)gridDim.x * blockDim.x) {
    const DInst& D = pool.insts[pool.part_inst[g]];
    const long long lp = g - D.part_off;
    const int32_t* rc = raw_cur + raw_rows_off[pool.part_inst[g]] + lp * D.SL;
    const int32_t* rp = raw_prev + raw_rows_off[pool.part_inst[g]] + lp * D.SL;
    int32_t* dc = pool.rows + D.rows_off + lp * D.SLP;
    int32_t* dp = pool.prev_rows + D.rows_off + lp * D.SLP;
    for (int i = 0; i < D.SLP; ++i) {
      dc[i] = i < D.SL ? rc[i] : BLANCE_NO_NODE;
      dp[i] = i < D.SL ? rp[i] : BLANCE_NO_NODE;
    }
    const uint8_t* sc = cur_shape + raw_shape_off[pool.part_inst[g]] + lp * D.S;
    const uint8_t* sp = prev_shape + raw_shape_off[pool.part_inst[g]] + lp * D.S;
    uint32_t mc = 0, mp = 0;
    for (int s = 0; s < D.S; ++s) { mc |= (uint32_t)(sc[s] & 3u) << (2 * s); mp |= (uint32_t)(sp[s] & 3u) << (2 * s); }
    pool.pmeta[g] = mc;
    pool.prev_meta[g] = mp;
  }
}

// ---- D2H side: device layout -> caller layout -------------------------------------------
__global__ void k_pack(DPool pool, int32_t* __restrict__ raw_next, uint8_t* __restrict__ next_shape,
                       uint8_t* __restrict__ warn, const long long* __restrict__ raw_rows_off,
                       const long long* __restrict__ raw_shape_off, long long n_parts_total) {
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n_parts_total;
       g += (long long)gridDim.x * blockDim.x) {
    const int inst = pool.part_inst[g];
    const DInst& D = pool.insts[inst];
    const long long lp = g - D.part_off;
    const int32_t* src = pool.rows + D.rows_off + lp * D.SLP;
    int32_t* dst = raw_next + raw_rows_off[inst] + lp * D.SL;
    for (int i = 0; i < D.SL; ++i) dst[i] = src[i];
    const uint32_t m = pool.pmeta[g];
    uint8_t* ds = next_shape + raw_shape_off[inst] + lp * D.S;
    uint8_t* dw = warn + raw_shape_off[inst] + lp * D.S;
    for (int s = 0; s < D.S; ++s) { ds[s] = (uint8_t)meta_shape(m, s); dw[s] = (uint8_t)((m >> (16 + s)) & 1u); }
  }
}

// ---- start of an iteration (plan.go:83-88, 70) -------------------------------------------
// Working rows = partitionsToAssign rows minus the to-be-removed nodes (order kept);
// every present state list becomes a non-nil slice; warnings are reset.
__global__ void k_prepare_rows(DPool pool, long long n_parts_total) {
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n_parts_total;
       g += (long long)gridDim.x * blockDim.x) {
    const DInst& D = pool.insts[pool.part_inst[g]];
    if (!D.active || !(pool.pflags[g] & PF_IN_ASSIGN)) continue;
    int32_t* row = pool.rows + D.rows_off + (g - D.part_off) * D.SLP;
    uint32_t m = pool.pmeta[g] & 0xFFFFu;          // drop the warn bits of the previous iteration
    for (int s = 0; s < D.S; ++s) {
      if (meta_shape(m, s) == BLANCE_SHAPE_ABSENT) continue;
      m = meta_set_shape(m, s, BLANCE_SHAPE_LIST);
      if (!D.rm_active) continue;
      int o = D.state_slot_off[s];
      const int hi = D.state_slot_off[s + 1];
      for (int i = o; i < hi; ++i) {
        const int32_t x = row[i];
        if (x == BLANCE_NO_NODE) break;
        if (!pool.node_removed[D.nodeid_off + x]) row[o++] = x;
      }
      for (; o < hi; ++o) row[o] = BLANCE_NO_NODE;
    }
    pool.pmeta[g] = m;
  }
}

// ---- countStateNodes (plan.go:374-399) over ALL of prevMap ---------------------------------
// Weighted histogram state x node.  SMEM_PRIV: one instance whose S*N table fits in
// shared memory -> per-CTA private histogram, flushed once (keeps 3M atomics off L2).
template <bool SMEM_PRIV>
__global__ void k_count_prev(DPool pool, long long n_parts_total) {
  extern __shared__ int32_t hist[];
  const DInst& D0 = pool.insts[0];
  const int table = SMEM_PRIV ? D0.S * D0.N : 0;
  if (SMEM_PRIV) {
    for (int i = threadIdx.x; i < table; i += blockDim.x) hist[i] = 0;
    __syncthreads();
  }
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n_parts_total;
       g += (long long)gridDim.x * blockDim.x) {
    const DInst& D = SMEM_PRIV ? D0 : pool.insts[pool.part_inst[g]];
    if (!D.active || !(pool.pflags[g] & PF_IN_PREV)) continue;
    const int32_t w = (D.has_part_weights && (pool.pflags[g] & PF_HAS_WEIGHT)) ? pool.pweight[g] : 1;
    const int32_t* row = pool.prev_rows + D.rows_off + (g - D.part_off) * D.SLP;
    for (int s = 0; s < D.S; ++s)
      for (int i = D.state_slot_off[s]; i < D.state_slot_off[s + 1]; ++i) {
        const int32_t x = row[i];
        if (x == BLANCE_NO_NODE) break;
        if (x >= D.N) continue;                       // a name outside nodesAll: never scored
        if (SMEM_PRIV) atomicAdd(&hist[s * D.N + x], w);
        else atomicAdd(&pool.counts[D.counts_off + (long long)s * D.N + x], w);
      }
  }
  if (SMEM_PRIV) {
    __syncthreads();
    for (int i = threadIdx.x; i < table; i += blockDim.x)
      if (hist[i]) atomicAdd(&pool.counts[D0.counts_off + i], hist[i]);
  }
}

// ---- partitionSorter key (plan.go:519-562) ----------------------------------------------------
// key = bucket(2) | 999999999 - weight (32) | name rank (30); partitions that are not being
// assigned sort to the end.
__global__ void k_build_keys(DPool pool, int s, long long n_parts_total) {
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n_parts_total;
       g += (long long)gridDim.x * blockDim.x) {
    const DInst& D = pool.insts[pool.part_inst[g]];
    pool.order_alt[g] = (int32_t)(g - D.part_off);
    const uint8_t f = pool.pflags[g];
    if (!D.active || s >= D.S || D.state_constraints[s] <= 0 || !(f & PF_IN_ASSIGN)) { pool.keys_alt[g] = ~0ull; continue; }
    const int32_t* row = pool.rows + D.rows_off + (g - D.part_off) * D.SLP;
    unsigned long long bucket = 2;
    bool b0 = false;
    if (D.rm_active && (f & PF_IN_PREV)) {
      const int32_t* prow = pool.prev_rows + D.rows_off + (g - D.part_off) * D.SLP;
      for (int i = D.state_slot_off[s]; i < D.state_slot_off[s + 1]; ++i) {
        const int32_t x = prow[i];
        if (x == BLANCE_NO_NODE) break;
        b0 |= pool.node_removed[D.nodeid_off + x] != 0;
      }
    }
    if (b0) bucket = 0;
    else if (!D.add_is_nil) {
      bool hit = false;
      if (D.add_active)
        for (int i = 0; i < D.SLP; ++i) {
          const int32_t x = row[i];
          if (x != BLANCE_NO_NODE) hit |= pool.node_added[D.nodeid_off + x] != 0;
        }
      if (!hit) bucket = 1;
    }
    const long long w = (D.has_part_weights && (f & PF_HAS_WEIGHT)) ? pool.pweight[g] : 1;
    const unsigned long long wkey = (unsigned long long)(999999999LL - w) & 0xFFFFFFFFull;   // plan.go:539
    pool.keys_alt[g] = (bucket << 62) | (wkey << 30) | (unsigned long long)(uint32_t)pool.name_rank[g];
  }
}

// ---- step stream of a pass: records in the sorted order, so the sequential kernel reads linearly -----
// record i of an instance (SLP + 8 words), pre-decoded so the chain does no per-step decoding:
//   row[SLP] | meta, w_p, top, partition | stickiness (double), n_cur, row_clean
// w_p = partition weight (plan.go:269-275), stickiness per plan.go:104-115, top = first node of the
// top-priority state or NU for "" (plan.go:134-138).
__global__ void k_gather_stream(DPool pool, int s, long long n_parts_total) {
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n_parts_total;
       g += (long long)gridDim.x * blockDim.x) {
    const DInst& D = pool.insts[pool.part_inst[g]];
    if (!D.active || s >= D.S || D.state_constraints[s] <= 0) continue;
    const long long i = g - D.part_off;                 // step index inside the instance
    if (i >= D.n_assign) continue;
    const int32_t p = pool.order[g];
    const int REC = D.SLP + 8;
    int32_t* dst = pool.stream + D.stream_off + i * REC;
    const int32_t* row = pool.rows + D.rows_off + (long long)p * D.SLP;
    for (int t = 0; t < D.SLP; ++t) dst[t] = row[t];
    const uint8_t f = pool.pflags[D.part_off + p];
    int32_t w_p = 1;
    double stick = 1.5;
    if (D.has_part_weights) {
      if (f & PF_HAS_WEIGHT) { w_p = pool.pweight[D.part_off + p]; stick = (double)w_p; }
      else if (D.state_has_stickiness[s]) stick = (double)D.state_stickiness[s];
    }
    int32_t top = D.NU;
    const int ts = D.state_slot_off[D.top_state];
    if (D.state_slot_off[D.top_state + 1] > ts && row[ts] != BLANCE_NO_NODE) top = row[ts];
    dst[D.SLP] = (int32_t)pool.pmeta[D.part_off + p];
    dst[D.SLP + 1] = w_p;
    dst[D.SLP + 2] = top;
    dst[D.SLP + 3] = p;
    const long long sb = __double_as_longlong(stick);
    dst[D.SLP + 4] = (int32_t)(sb & 0xFFFFFFFFll);
    dst[D.SLP + 5] = (int32_t)(sb >> 32);
    // the current list of state s: its length, and whether it is "clean" (nodes distinct, inside
    // nodesAll, and listed under no other state of this row) - the sticky fast path needs both
    const int lo = D.state_slot_off[s], hi = D.state_slot_off[s + 1];
    int n_cur = 0;
    bool clean = true;
    for (int a = lo; a < hi && row[a] != BLANCE_NO_NODE; ++a) {
      ++n_cur;
      if (row[a] >= D.N) clean = false;
      for (int b = 0; b < D.SL; ++b)
        if (b != a && row[b] == row[a]) clean = false;
    }
    dst[D.SLP + 6] = n_cur;
    dst[D.SLP + 7] = clean ? 1 : 0;
    pool.srank[g] = 0;
    if (clean && n_cur == D.state_constraints[s]) atomicAdd(&pool.insts[pool.part_inst[g]].n_elig, 1);
    if (clean && n_cur <= D.state_constraints[s]) atomicAdd(&pool.insts[pool.part_inst[g]].n_clean, 1);
  }
}

// ---- the all-sticky hypothesis of the speculative pass (assign_pass_spec.cuh) -----------------------------
// If every eligible step (clean row, exactly k current nodes) kept its nodes, step i would find
// nodeToNodeCounts[top][c] = the number of EARLIER eligible steps of the pass with the same (top, c) pair.
// k_pair_keys emits one (pair, item) per eligible step and current node, a stable radix sort groups the pairs
// (items of a pair stay in step order), k_pair_rank turns the position inside the group into qstat[step][q].
__global__ void k_pair_keys(DPool pool, int s, long long n_parts_total, int inst_shift) {
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n_parts_total;
       g += (long long)gridDim.x * blockDim.x) {
    const int inst = pool.part_inst[g];
    const DInst& D = pool.insts[inst];
    unsigned long long key[4] = {~0ull, ~0ull, ~0ull, ~0ull};
    const long long i = g - D.part_off;
    if (D.active && s < D.S && D.pass_mode == 2 && i < D.n_assign) {
      const int REC = D.SLP + 8, k = D.state_constraints[s];
      const int32_t* rec = pool.stream + D.stream_off + i * REC;
      if (rec[D.SLP + 7] != 0 && rec[D.SLP + 6] == k) {
        const unsigned long long hi = ((unsigned long long)(uint32_t)inst << inst_shift) | ((unsigned long long)(uint32_t)rec[D.SLP + 2] << 13);
        for (int q = 0; q < k && q < 4; ++q) key[q] = hi | (unsigned long long)(uint32_t)rec[D.state_slot_off[s] + q];
      }
    }
    for (int q = 0; q < 4; ++q) {
      pool.pair_keys_alt[4 * g + q] = key[q];
      pool.pair_vals_alt[4 * g + q] = (uint32_t)(4 * g + q);
      pool.qstat[4 * g + q] = 0;
    }
  }
}

__global__ void k_pair_rank(DPool pool, long long n_items) {
  for (long long x = blockIdx.x * (long long)blockDim.x + threadIdx.x; x < n_items; x += (long long)gridDim.x * blockDim.x) {
    const unsigned long long key = pool.pair_keys[x];
    if (key == ~0ull) continue;
    long long lo = 0, hi = x;                  // first position holding `key` (keys are sorted)
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (pool.pair_keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    pool.qstat[pool.pair_vals[x]] = (int32_t)(x - lo);
  }
}

// Which kernel runs the pass of state s for each instance (one thread per instance): the sequencer
// kernel pays off when many rows can be decided by the sticky test; it needs k <= 4, no hierarchy
// rules for the state, and a node mirror that fits in shared memory.
__global__ void k_pick_mode(DPool pool, int s, int n_inst, int seq_allowed, int spec_allowed, int spec_max_n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_inst) return;
  DInst& D = pool.insts[i];
  int mode = 0;
  if (D.active && s < D.S && D.state_constraints[s] > 0) {
    const bool rules = D.has_hier_rules && D.rule_off[s + 1] > D.rule_off[s];
    const bool shape_ok = !rules && D.state_constraints[s] <= 4 && D.SLP <= 8 && D.n_assign >= 64 && 4ll * D.n_elig >= (long long)D.n_assign;
    if (seq_allowed && (D.engine == BLANCE_ENGINE_AUTO || D.engine == BLANCE_ENGINE_SEQUENCER) && shape_ok && D.N <= 4096) mode = 1;
    // the speculative kernel resolves clean rows with at most k current nodes on its own; anything else costs a
    // full team evaluation, so it wants nearly all rows clean
    if (spec_allowed && D.engine == BLANCE_ENGINE_AUTO && shape_ok && D.N <= spec_max_n &&
        64ll * D.n_clean >= 63ll * (long long)D.n_assign)
      mode = 2;
  }
  D.pass_mode = mode;
  D.n_elig = 0;
  D.n_clean = 0;
}

// After the pass: rebuild every partition's row from the step's outcome (plan.go:290-301), in
// parallel.  ostream record i = { chosen[0..k), n_chosen }; stream record i still
// holds the row / meta / partition the step started from.
__global__ void k_scatter_stream(DPool pool, int s, long long n_parts_total) {
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n_parts_total;
       g += (long long)gridDim.x * blockDim.x) {
    const DInst& D = pool.insts[pool.part_inst[g]];
    if (!D.active || s >= D.S || D.state_constraints[s] <= 0) continue;
    const long long i = g - D.part_off;
    if (i >= D.n_assign) continue;
    const int REC = D.SLP + 8, k = D.state_constraints[s];
    const int32_t* in = pool.stream + D.stream_off + i * REC;
    const int32_t* out_rec = pool.ostream + D.stream_off + i * REC;
    const int32_t p = in[D.SLP + 3];
    const uint32_t meta = (uint32_t)in[D.SLP];
    const int lo_s = D.state_slot_off[s], hi_s = D.state_slot_off[s + 1];
    // a step the speculative kernel accepted as sticky keeps its k current nodes, in (score, position) order:
    // srank = 0x80 | rank of current node q in bits 2q..2q+1.  With k = 4 the flag shares bit 7 with the rank of the
    // last node, so that rank is taken from the others: the ranks are a permutation of 0..k-1
    const uint32_t sr = pool.srank[g];
    int32_t sticky_out[4];
    if (sr & 0x80u) {
      uint32_t rank_sum = 0;
      for (int q = 0; q + 1 < k && q < 3; ++q) {
        const uint32_t r = (sr >> (2 * q)) & 3u;
        sticky_out[r] = in[lo_s + q];
        rank_sum += r;
      }
      if (k >= 1 && k <= 4) sticky_out[(uint32_t)(k * (k - 1) / 2) - rank_sum] = in[lo_s + k - 1];
    }
    const int32_t* out = (sr & 0x80u) ? sticky_out : out_rec;
    const int n_chosen = (sr & 0x80u) ? k : out_rec[k];
    int32_t* row = pool.rows + D.rows_off + (long long)p * D.SLP;
    uint32_t nmeta = meta;
    bool have_higher_key = false;
    for (int s2 = 0; s2 < D.S; ++s2) {
      if (meta_shape(meta, s2) == BLANCE_SHAPE_ABSENT) continue;
      if (D.state_priority[s2] < D.state_priority[s]) have_higher_key = true;
      if (s2 == s) continue;
      nmeta = meta_set_shape(nmeta, s2, BLANCE_SHAPE_LIST);          // misc.go:29: non-nil after removal
      int o = D.state_slot_off[s2];
      const int e = D.state_slot_off[s2 + 1];
      for (int sl = o; sl < e; ++sl) {                               // removeNodesFromNodesByState x2
        const int32_t x = in[sl];
        if (x == BLANCE_NO_NODE) break;
        bool rm = false;
        for (int q = lo_s; q < hi_s && in[q] != BLANCE_NO_NODE; ++q) rm |= (in[q] == x);
        for (int c = 0; c < n_chosen; ++c) rm |= (out[c] == x);
        if (!rm) row[o++] = x;
      }
      for (; o < e; ++o) row[o] = BLANCE_NO_NODE;
    }
    for (int sl = lo_s; sl < hi_s; ++sl) row[sl] = (sl - lo_s) < n_chosen ? out[sl - lo_s] : BLANCE_NO_NODE;   // plan.go:299
    // nil result: candidateNodes stays nil only if nodesNext is empty, no higher-priority key filtered
    // it and the hierarchy block did not run (plan.go:142,149-150,225)
    const bool nil = n_chosen == 0 && D.n_valid == 0 && !have_higher_key && !D.has_hier_rules;
    nmeta = meta_set_shape(nmeta, s, nil ? BLANCE_SHAPE_NIL : BLANCE_SHAPE_LIST);
    if (n_chosen < k) nmeta |= 1u << (16 + s);                       // plan.go:228-235
    pool.pmeta[D.part_off + p] = nmeta;
  }
}

// ---- convergence test (plan.go:36-42) -------------------------------------------------------------
__global__ void k_compare(DPool pool, long long n_parts_total) {
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n_parts_total;
       g += (long long)gridDim.x * blockDim.x) {
    DInst& D = pool.insts[pool.part_inst[g]];
    const uint8_t f = pool.pflags[g];
    if (!D.active || !(f & PF_IN_ASSIGN)) continue;
    // (a prevMap entry with keys outside the model never equals the new partition: reflect.DeepEqual, plan.go:38)
    bool same = (f & PF_IN_PREV) && !(f & PF_PREV_EXTRA) && ((pool.pmeta[g] & 0xFFFFu) == (pool.prev_meta[g] & 0xFFFFu));
    if (same) {
      const int32_t* a = pool.rows + D.rows_off + (g - D.part_off) * D.SLP;
      const int32_t* b = pool.prev_rows + D.rows_off + (g - D.part_off) * D.SLP;
      for (int i = 0; i < D.SLP; ++i) same &= (a[i] == b[i]);
    }
    if (!same) D.mismatch = 1;
  }
}

// ---- plan.go:49-52: prevMap[p] = partitionsToAssign[p] = next[p] --------------------------------------
__global__ void k_commit(DPool pool, long long n_parts_total) {
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n_parts_total;
       g += (long long)gridDim.x * blockDim.x) {
    const DInst& D = pool.insts[pool.part_inst[g]];
    const uint8_t f = pool.pflags[g];
    if (!D.active || !D.mismatch || !(f & PF_IN_ASSIGN)) continue;
    const int32_t* a = pool.rows + D.rows_off + (g - D.part_off) * D.SLP;
    int32_t* b = pool.prev_rows + D.rows_off + (g - D.part_off) * D.SLP;
    for (int i = 0; i < D.SLP; ++i) b[i] = a[i];
    pool.prev_meta[g] = pool.pmeta[g] & 0xFFFFu;
    pool.pflags[g] = (uint8_t)((f | PF_IN_PREV) & ~PF_PREV_EXTRA);
  }
}

// ---- loop control of plan.go:32-56, one thread per instance --------------------------------------------
__global__ void k_next_iter(DPool pool, int n_inst, int* any_active) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_inst) return;
  DInst& D = pool.insts[i];
  if (!D.active) return;
  D.iters_run += 1;
  if (!D.mismatch) { D.converged = 1; D.active = 0; return; }
  D.converged = 0;
  if (D.iters_run >= D.max_iters) { D.active = 0; return; }
  D.mismatch = 0;
  D.rm_active = 0;           // nodesToRemove = []string{}
  D.add_active = 0;          // nodesToAdd = []string{} (non-nil: everyone lands in bucket "1")
  D.add_is_nil = 0;
  D.use_rest = 1;
  D.P = D.PU;                // len(prevMap) after plan.go:49-52
  atomicAdd(any_active, 1);
}

// ---- CalcPartitionMoves (moves.go:41-136), one thread per partition ------------------------------------------
__global__ void k_calc_moves(int32_t n_parts, int32_t n_states, int32_t n_visit, const int32_t* __restrict__ slot_off,
                             const int32_t* __restrict__ beg_rows, const int32_t* __restrict__ end_rows,
                             int32_t favor_min, int32_t max_ops, int32_t* __restrict__ op_node,
                             uint8_t* __restrict__ op_state, uint8_t* __restrict__ op_kind,
                             int32_t* __restrict__ op_count) {
  const int SL = slot_off[n_states];
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < n_parts;
       p += (long long)gridDim.x * blockDim.x) {
    const int32_t* beg = beg_rows + p * SL;
    const int32_t* end = end_rows + p * SL;
    int32_t* on = op_node + p * max_ops;
    uint8_t* os = op_state + p * max_ops;
    uint8_t* ok = op_kind + p * max_ops;
    int cnt = 0;
    auto in_row = [&](const int32_t* row, int32_t node) { bool r = false; for (int i = 0; i < SL; ++i) r |= (row[i] == node); return r; };
    auto emit = [&](int32_t node, int st, int kind) {                 // addMoves + seen, moves.go:51-58
      for (int j = 0; j < cnt; ++j) if (on[j] == node) return;
      if (cnt < max_ops) { on[cnt] = node; os[cnt] = (uint8_t)st; ok[cnt] = (uint8_t)kind; ++cnt; }
    };
    for (int step = 0; step < n_visit; ++step) {
      const int si = favor_min ? n_visit - 1 - step : step;
      const int lo = slot_off[si], hi = slot_off[si + 1];
      for (int phase = 0; phase < 4; ++phase) {
        // !favorMinNodes: promote, demote, add, del (moves.go:66-90); favorMinNodes: del, demote, promote, add (:92-116)
        const int what = favor_min ? (phase == 0 ? 3 : phase == 1 ? 1 : phase == 2 ? 0 : 2) : phase;
        if (what <= 1) {                      // findStateChanges, moves.go:121-136
          const int jlo = what == 0 ? si + 1 : 0, jhi = what == 0 ? n_visit : si;
          for (int i = lo; i < hi && end[i] != BLANCE_NO_NODE; ++i)
            for (int j = jlo; j < jhi; ++j)
              for (int b = slot_off[j]; b < slot_off[j + 1] && beg[b] != BLANCE_NO_NODE; ++b)
                if (beg[b] == end[i]) emit(end[i], si, what == 0 ? BLANCE_OP_PROMOTE : BLANCE_OP_DEMOTE);
        } else if (what == 2) {               // end[s] \ beg[s], restricted to adds = endAll \ begAll
          for (int i = lo; i < hi && end[i] != BLANCE_NO_NODE; ++i)
            if (!in_row(beg, end[i])) emit(end[i], si, BLANCE_OP_ADD);
        } else {                              // beg[s] \ end[s], restricted to dels = begAll \ endAll
          for (int i = lo; i < hi && beg[i] != BLANCE_NO_NODE; ++i)
            if (!in_row(end, beg[i])) emit(beg[i], BLANCE_OP_STATE_NONE, BLANCE_OP_DEL);
        }
      }
    }
    op_count[p] = cnt;
  }
}

// ---- move lists for the orchestrator: CSR compaction and one round of findAvailableMovesUnlocked -----------------
__global__ void k_moves_compact(int32_t n_parts, int32_t max_ops, const long long* __restrict__ op_off,
                                const int32_t* __restrict__ op_count, const int32_t* __restrict__ in_node,
                                const uint8_t* __restrict__ in_state, const uint8_t* __restrict__ in_kind,
                                int32_t* __restrict__ out_node, uint8_t* __restrict__ out_state, uint8_t* __restrict__ out_kind) {
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < n_parts; p += (long long)gridDim.x * blockDim.x) {
    const long long o = op_off[p];
    for (int j = 0; j < op_count[p]; ++j) {
      out_node[o + j] = in_node[p * max_ops + j];
      out_state[o + j] = in_state[p * max_ops + j];
      out_kind[o + j] = in_kind[p * max_ops + j];
    }
  }
}

__device__ __forceinline__ int move_op_weight(int kind) {           // MoveOpWeight, orchestrate.go:189-194
  return kind == BLANCE_OP_PROMOTE ? 1 : kind == BLANCE_OP_DEMOTE ? 2 : kind == BLANCE_OP_ADD ? 3 : 4;
}

// per partition: the node of its next move (orchestrate.go:755-757) as a sort key; per node: how many, and the
// lowest (MoveOpWeight, partition) (orchestrate.go:177-186 with a fixed tie order)
__global__ void k_moves_next(int32_t n_parts, int32_t n_node_ids, const long long* __restrict__ op_off,
                             const int32_t* __restrict__ op_node, const uint8_t* __restrict__ op_kind,
                             const int32_t* __restrict__ next, uint32_t* __restrict__ key, int32_t* __restrict__ val,
                             int32_t* __restrict__ node_cnt, unsigned long long* __restrict__ node_best) {
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < n_parts; p += (long long)gridDim.x * blockDim.x) {
    uint32_t k = 0xFFFFFFFFu;
    const long long n_ops = op_off[p + 1] - op_off[p];
    const int32_t nx = next[p];
    if (nx >= 0 && nx < n_ops) {
      const int32_t node = op_node[op_off[p] + nx];
      if (node >= 0 && node < n_node_ids) {
        k = (uint32_t)node;
        atomicAdd(&node_cnt[node], 1);
        atomicMin(&node_best[node], ((unsigned long long)move_op_weight(op_kind[op_off[p] + nx]) << 32) | (uint32_t)p);
      }
    }
    key[p] = k;
    val[p] = (int32_t)p;
  }
}

__global__ void k_moves_best(int32_t n_node_ids, const unsigned long long* __restrict__ node_best, int32_t* __restrict__ best_part) {
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < n_node_ids; n += gridDim.x * blockDim.x)
    best_part[n] = node_best[n] == ~0ull ? -1 : (int32_t)(node_best[n] & 0xFFFFFFFFull);
}

}  // namespace blance_dev
