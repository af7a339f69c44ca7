// blance_b200/csrc/c_abi.cu — the C ABI of libblance_b200.so (include/blance_b200.h):
// validation, pooling of a batch of plan instances into one set of device arrays,
// the host side of the convergence loop (plan.go:32-56) and the launches.
// No CPU fallback: every compute entry point needs a CUDA device.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_radix_sort.cuh>

#include "assign_pass.cuh"
#include "assign_pass_seq.cuh"
#include "assign_pass_spec.cuh"
#include "aux_kernels.cuh"
#include "blance_b200.h"
#include "device_types.cuh"

using namespace blance_dev;

static std::string g_create_error;

// Opted-in dynamic shared memory of k_assign_pass_seq<1|2|4|8>, per device.  The attribute belongs to the
// (function, device) pair, not to a blance_ctx, and must only ever be raised.
static std::mutex g_seq_dyn_mu;
static size_t g_seq_dyn[64][4][4];   // [device][NPT index][K - 1]
static size_t g_spec_dyn[64][4];     // [device][K - 1], k_assign_pass_spec

struct blance_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  std::string err;
  std::mutex mu;
  void* cub_tmp = nullptr;
  size_t cub_tmp_bytes = 0;
  std::vector<cudaEvent_t> events;   // pool for pass timing
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  int* d_any_active = nullptr;
  int* h_any_active = nullptr;       // pinned
  long long launches = 0;            // kernels of this library launched so far
  void* h_stage = nullptr;           // pinned staging of a batch (kept between calls, grow-only)
  size_t h_stage_bytes = 0;
  std::vector<blance_ctx*> children; // blance_ctx_create_multi: one single-device context per GPU
};

#define CK(call)                                                                           \
  do {                                                                                     \
    cudaError_t e_ = (call);                                                               \
    if (e_ != cudaSuccess) {                                                               \
      char b_[512];                                                                        \
      std::snprintf(b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      ctx->err = b_;                                                                       \
      return BLANCE_ERR_CUDA;                                                              \
    }                                                                                      \
  } while (0)

static int fail(blance_ctx* ctx, int st, const std::string& msg) {
  if (ctx) ctx->err = msg; else g_create_error = msg;
  return st;
}

extern "C" int blance_version(void) { return 100; }

extern "C" int64_t blance_ctx_kernel_launches(const blance_ctx* ctx) {
  if (!ctx) return 0;
  long long n = ctx->launches;
  for (const blance_ctx* c : ctx->children) n += c->launches;
  return n;
}

extern "C" int blance_ctx_device_count(const blance_ctx* ctx) { return !ctx ? 0 : ctx->children.empty() ? 1 : (int)ctx->children.size(); }

extern "C" const char* blance_last_error(const blance_ctx* ctx) {
  return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

extern "C" int blance_ctx_create(blance_ctx** out, int device_id) {
  if (!out) return fail(nullptr, BLANCE_ERR_INVALID_ARG, "blance_ctx_create: out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0)
    return fail(nullptr, BLANCE_ERR_CUDA, std::string("no CUDA device available (") +
                                              (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                                              "); libblance_b200 has no CPU fallback");
  if (device_id < 0) {
    if (cudaGetDevice(&device_id) != cudaSuccess) device_id = 0;
  }
  if (device_id >= count) return fail(nullptr, BLANCE_ERR_INVALID_ARG, "blance_ctx_create: device id out of range");
  blance_ctx* ctx = new blance_ctx();
  ctx->device = device_id;
  auto bail = [&](const char* what, cudaError_t er) {
    std::string msg = std::string(what) + ": " + cudaGetErrorString(er);
    delete ctx;
    return fail(nullptr, BLANCE_ERR_CUDA, msg);
  };
  if ((e = cudaSetDevice(device_id)) != cudaSuccess) return bail("cudaSetDevice", e);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device_id)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
  ctx->sm_count = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
  for (auto& ev : ctx->ev)
    if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail("cudaEventCreate", e);
  {
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device_id) == cudaSuccess) {
      unsigned long long keep = ~0ull;              // keep freed arenas cached in the pool between calls
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
  }
  if ((e = cudaMalloc(&ctx->d_any_active, sizeof(int))) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = cudaMallocHost(&ctx->h_any_active, sizeof(int))) != cudaSuccess) return bail("cudaMallocHost", e);
  *out = ctx;
  return BLANCE_OK;
}

// One context over several GPUs of the node (SURVEY.md section 8b: blance_ctx_create(gpu_ids, n_gpus)).  A batch
// (blance_plan_next_map_batch) is sharded instance i -> device i mod n, one host thread per device, no collective:
// plan instances are independent.  Everything else runs on the first device.
extern "C" int blance_ctx_create_multi(blance_ctx** out, const int* device_ids, int n_devices) {
  if (!out) return fail(nullptr, BLANCE_ERR_INVALID_ARG, "blance_ctx_create_multi: out is NULL");
  *out = nullptr;
  if (!device_ids || n_devices <= 0) return fail(nullptr, BLANCE_ERR_INVALID_ARG, "blance_ctx_create_multi: no devices given");
  for (int a = 0; a < n_devices; ++a)
    for (int b = 0; b < a; ++b)
      if (device_ids[a] == device_ids[b]) return fail(nullptr, BLANCE_ERR_INVALID_ARG, "blance_ctx_create_multi: a device is listed twice");
  blance_ctx* parent = new blance_ctx();
  for (int a = 0; a < n_devices; ++a) {
    blance_ctx* c = nullptr;
    const int st = blance_ctx_create(&c, device_ids[a]);
    if (st != BLANCE_OK) {
      for (blance_ctx* k : parent->children) blance_ctx_destroy(k);
      delete parent;
      return st;                       // g_create_error already says why
    }
    parent->children.push_back(c);
  }
  parent->device = parent->children[0]->device;
  parent->sm_count = parent->children[0]->sm_count;
  *out = parent;
  return BLANCE_OK;
}

extern "C" void blance_ctx_destroy(blance_ctx* ctx) {
  if (!ctx) return;
  if (!ctx->children.empty()) {
    for (blance_ctx* c : ctx->children) blance_ctx_destroy(c);
    delete ctx;
    return;
  }
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  for (auto ev : ctx->events) cudaEventDestroy(ev);
  for (auto ev : ctx->ev) if (ev) cudaEventDestroy(ev);
  if (ctx->cub_tmp) cudaFree(ctx->cub_tmp);
  if (ctx->d_any_active) cudaFree(ctx->d_any_active);
  if (ctx->h_any_active) cudaFreeHost(ctx->h_any_active);
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

// ---------------------------------------------------------------------------------------
// A batch of instances resident on the device.

struct blance_plan {
  int n_inst = 0;
  std::vector<DInst> h_insts;          // initial descriptors (dynamic fields at their start values)
  std::vector<long long> raw_rows_off, raw_shape_off;   // caller-layout offsets per instance
  long long PT = 0, RT = 0, NT = 0, NUT = 0, CT = 0, N2T = 0, MT = 0, RRT = 0, RST = 0, ST = 0;
  int max_N = 0, max_S = 0, max_NU = 0;
  int pair_inst_shift = 0, pair_end_bit = 64;   // key layout of the (top, node) pair sort (k_pair_keys)
  bool any_state_active[BL_S_MAX] = {};
  void* arena = nullptr;               // one device allocation, carved below
  size_t arena_bytes = 0;
  DPool pool{};
  // immutable copies of the mutable state, to replay the plan (blance_plan_run)
  int32_t *rows_init = nullptr, *prev_rows_init = nullptr;
  uint32_t *pmeta_init = nullptr, *prev_meta_init = nullptr;
  uint8_t* pflags_init = nullptr;
  // device staging in caller layout
  int32_t *raw_a = nullptr, *raw_b = nullptr;           // cur/prev rows in, next rows out (raw_a)
  uint8_t *rawsh_a = nullptr, *rawsh_b = nullptr;       // cur/prev shape in, next shape (a) / warn (b) out
  long long *d_raw_rows_off = nullptr, *d_raw_shape_off = nullptr;
  int* d_seg_off = nullptr;            // [n_inst+1] partition offsets for the segmented sort
  // pinned host staging (batch concatenation and results)
  void* h_stage = nullptr;
  size_t h_stage_bytes = 0;
  float last_kernel_ms = 0, last_pass_ms = 0;
  int pass_launches = 0;
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// sizes, pointers and limits of one instance (no table contents: those are blance_plan_in_check's)
static int check_structure(const blance_plan_in* in, std::string& why) {
  auto bad = [&](const char* what, int st = BLANCE_ERR_INVALID_ARG) {
    why = what;
    return st;
  };
  if (!in) return bad("plan_in is NULL");
  if (in->n_nodes < 0 || in->n_node_ids < in->n_nodes || in->n_states < 0 || in->n_parts < 0 || in->n_slots < 0)
    return bad("negative size or n_node_ids < n_nodes");
  if (in->n_states > BL_S_MAX) return bad("more than 8 model states", BLANCE_ERR_UNSUPPORTED);
  if (in->n_slots > BL_SLP_MAX) return bad("more than 32 slots per row", BLANCE_ERR_UNSUPPORTED);
  if (in->n_nodes > 8192) return bad("more than 8192 nodes", BLANCE_ERR_UNSUPPORTED);   /* 512 compute threads x 16 nodes */
  if (in->n_states > 0 && (!in->state_priority || !in->state_constraints || !in->state_slot_off ||
                           !in->state_stickiness || !in->state_has_stickiness))
    return bad("state tables are NULL");
  if (in->n_states > 0 && (in->top_state < 0 || in->top_state >= in->n_states)) return bad("top_state out of range");
  if (in->n_states > 0 && in->state_slot_off[in->n_states] != in->n_slots) return bad("state_slot_off[S] != n_slots");
  for (int s = 0; s < in->n_states; ++s) {
    if (in->state_slot_off[s + 1] < in->state_slot_off[s]) return bad("state_slot_off not monotone");
    if (in->state_constraints[s] > BL_K_MAX) return bad("constraints > 16", BLANCE_ERR_UNSUPPORTED);
    if (in->state_constraints[s] > in->state_slot_off[s + 1] - in->state_slot_off[s])
      return bad("a state's slot range is smaller than its constraints");
  }
  if (in->n_parts > 0 && (!in->part_in_prev || !in->part_in_assign || !in->part_weight || !in->part_has_weight ||
                          !in->part_name_rank))
    return bad("partition tables are NULL");
  if (in->n_parts > 0 && in->n_states > 0 && (!in->prev_shape || !in->cur_shape)) return bad("shape tables are NULL");
  if (in->n_parts > 0 && in->n_slots > 0 && (!in->prev_rows || !in->cur_rows)) return bad("row tables are NULL");
  if (in->n_node_ids > 0 && (!in->node_removed || !in->node_added)) return bad("node flag tables are NULL");
  if (in->n_nodes > 0 && in->has_node_weights && (!in->node_weight || !in->node_has_weight)) return bad("node weight tables are NULL");
  if (in->n_parts >= (1 << 30)) return bad("2^30 or more partitions", BLANCE_ERR_UNSUPPORTED);
  if (in->has_hier_rules) {
    if (!in->rule_off) return bad("rule_off is NULL");
    if (in->n_rules > 0 && !in->ie_mask) return bad("ie_mask is NULL");
    if (in->n_hier_bits < in->n_nodes) return bad("n_hier_bits < n_nodes");
    if ((in->n_hier_bits + 31) / 32 > 128) return bad("hierarchy universe above 4096 bits", BLANCE_ERR_UNSUPPORTED);
    for (int s = 0; s < in->n_states; ++s)
      if ((in->rule_off[s + 1] - in->rule_off[s]) * std::max(0, in->state_constraints[s]) > BL_PICK_MAX)
        return bad("rules x constraints > 32 for one state", BLANCE_ERR_UNSUPPORTED);
  }
  if (in->engine != BLANCE_ENGINE_AUTO && in->engine != BLANCE_ENGINE_LOCKSTEP && in->engine != BLANCE_ENGINE_SEQUENCER) return bad("unknown engine", BLANCE_ERR_UNSUPPORTED);
  if (in->booster_kind != BLANCE_BOOSTER_NONE && in->booster_kind != BLANCE_BOOSTER_CBGT_MAX)
    return bad("unknown booster_kind", BLANCE_ERR_UNSUPPORTED);
  return BLANCE_OK;
}

static int validate(blance_ctx* ctx, const blance_plan_in* in, int idx) {
  std::string why;
  const int st = check_structure(in, why);
  if (st == BLANCE_OK) return st;
  char b[256];
  std::snprintf(b, sizeof b, "instance %d: %s", idx, why.c_str());
  return fail(ctx, st, b);
}

/* The contents of the tables, for bindings that do not trust their own marshalling (the planning entry points
 * check sizes, pointers and limits only: a scan of every row would sit in the timed path of every call). */
extern "C" int blance_plan_in_check(const blance_plan_in* in, char* msg, int32_t msg_cap) {
  std::string why;
  auto done = [&](int st) {
    if (msg && msg_cap > 0) std::snprintf(msg, (size_t)msg_cap, "%s", why.c_str());
    return st;
  };
  int st = check_structure(in, why);
  if (st != BLANCE_OK) return done(st);
  auto bad = [&](const std::string& what, int code = BLANCE_ERR_INVALID_ARG) { why = what; return done(code); };
  if (in->n_states > 0 && in->state_slot_off[0] != 0) return bad("state_slot_off[0] != 0");
  const long long P = in->n_parts, SL = in->n_slots, S = in->n_states;
  for (int which = 0; which < 2; ++which) {
    const int32_t* rows = which ? in->cur_rows : in->prev_rows;
    const uint8_t* shape = which ? in->cur_shape : in->prev_shape;
    const char* name = which ? "cur" : "prev";
    int32_t lo = 0, hi = -1;
    for (long long i = 0; i < P * SL; ++i) { lo = std::min(lo, rows[i]); hi = std::max(hi, rows[i]); }
    if (lo < BLANCE_NO_NODE || hi >= in->n_node_ids)
      return bad(std::string(name) + "_rows holds a node id outside [-1, n_node_ids)");
    uint8_t sh = 0;
    for (long long i = 0; i < P * S; ++i) sh = std::max(sh, shape[i]);
    if (sh > BLANCE_SHAPE_LIST) return bad(std::string(name) + "_shape holds a value above BLANCE_SHAPE_LIST");
    // a state's list is filled from the left: no node after an empty slot
    for (long long p = 0; p < P; ++p)
      for (int s = 0; s < in->n_states; ++s) {
        bool gap = false;
        for (int c = in->state_slot_off[s]; c < in->state_slot_off[s + 1]; ++c) {
          const int32_t x = rows[p * SL + c];
          if (x == BLANCE_NO_NODE) gap = true;
          else if (gap) return bad(std::string(name) + "_rows: partition " + std::to_string(p) + " has a node after an empty slot of state " + std::to_string(s));
        }
      }
  }
  {
    // part_name_rank: 0 <= rank < 2^30, unique (it is the last word of the partition sort key, plan.go:512-528)
    std::vector<uint64_t> seen;
    std::vector<int32_t> big;
    seen.assign((size_t)((P + 63) / 64), 0);
    for (long long p = 0; p < P; ++p) {
      const int32_t r = in->part_name_rank[p];
      if (r < 0 || r >= (1 << 30)) return bad("part_name_rank outside [0, 2^30) at partition " + std::to_string(p));
      if (r < P) {
        if (seen[(size_t)(r >> 6)] >> (r & 63) & 1ull) return bad("part_name_rank " + std::to_string(r) + " appears twice");
        seen[(size_t)(r >> 6)] |= 1ull << (r & 63);
      } else big.push_back(r);
    }
    std::sort(big.begin(), big.end());
    if (std::adjacent_find(big.begin(), big.end()) != big.end()) return bad("a part_name_rank appears twice");
    // the weight word of the key is 999999999 - w printed with %10d (plan.go:539): beyond 999999999 the reference's
    // STRING order and a numeric order part ways
    for (long long p = 0; p < P; ++p)
      if (in->has_part_weights && in->part_has_weight[p] && in->part_weight[p] > 999999999)
        return bad("partition weight above 999999999 at partition " + std::to_string(p), BLANCE_ERR_UNSUPPORTED);
  }
  if (in->has_hier_rules)
    for (int s = 0; s <= in->n_states; ++s) {
      if (in->rule_off[s] < 0 || in->rule_off[s] > in->n_rules || (s > 0 && in->rule_off[s] < in->rule_off[s - 1]))
        return bad("rule_off is not a monotone offset table into the rules");
    }
  why.clear();
  return done(BLANCE_OK);
}

static void plan_release(blance_plan* pl, blance_ctx* ctx = nullptr) {
  if (!pl) return;
  if (pl->arena) {
    if (ctx) cudaFreeAsync(pl->arena, ctx->stream);     // back to the pool (stream ordered)
    else cudaFree(pl->arena);
  }
  delete pl;                         // (the pinned staging buffer belongs to the context)
}

static int grid_for(const blance_ctx* ctx, long long n, int block) {
  long long want = (n + block - 1) / block;
  long long cap = (long long)ctx->sm_count * 8;      // multiples of the SM count; kernels are grid-stride
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  return (int)want;
}

static int upload(blance_ctx* ctx, int n, const blance_plan_in* ins, blance_plan** out_plan) {
  *out_plan = nullptr;
  if (n <= 0) return fail(ctx, BLANCE_ERR_INVALID_ARG, "batch size must be positive");
  for (int i = 0; i < n; ++i) {
    int st = validate(ctx, &ins[i], i);
    if (st != BLANCE_OK) return st;
  }
  CK(cudaSetDevice(ctx->device));
  {
    cudaError_t stale = cudaGetLastError();      // never let an earlier, unrelated error be blamed on this call
    if (stale != cudaSuccess) return fail(ctx, BLANCE_ERR_CUDA, std::string("a previous CUDA call on this thread failed: ") + cudaGetErrorString(stale));
  }
  blance_plan* pl = new blance_plan();
  pl->n_inst = n;
  pl->h_insts.resize(n);
  pl->raw_rows_off.resize(n + 1);
  pl->raw_shape_off.resize(n + 1);
  std::vector<int> seg_off(n + 1);
  for (int i = 0; i < n; ++i) {
    const blance_plan_in& in = ins[i];
    DInst& D = pl->h_insts[i];
    std::memset(&D, 0, sizeof D);
    D.N = in.n_nodes; D.NU = in.n_node_ids; D.S = in.n_states; D.PU = in.n_parts; D.SL = in.n_slots;
    D.SLP = std::max(4, (int)align_up((size_t)in.n_slots, 4));
    D.HW = in.has_hier_rules ? (in.n_hier_bits + 31) / 32 : 0;
    D.n_rules = in.has_hier_rules ? in.n_rules : 0;
    D.top_state = in.top_state; D.booster = in.booster_kind;
    D.has_part_weights = in.has_part_weights; D.has_node_weights = in.has_node_weights;
    D.has_hier_rules = in.has_hier_rules; D.max_iters = in.max_iters; D.engine = in.engine;
    D.debug = getenv("BLANCE_SPEC_STATS") ? 1 : 0;
    for (int s = 0; s < in.n_states; ++s) {
      D.state_priority[s] = in.state_priority[s];
      D.state_constraints[s] = in.state_constraints[s];
      D.state_slot_off[s] = in.state_slot_off[s];
      D.state_stickiness[s] = in.state_stickiness[s];
      D.state_has_stickiness[s] = in.state_has_stickiness[s];
      D.rule_off[s] = in.has_hier_rules ? in.rule_off[s] : 0;
      if (in.state_constraints[s] > 0) pl->any_state_active[s] = true;
    }
    D.state_slot_off[in.n_states] = in.n_slots;
    D.rule_off[in.n_states] = in.has_hier_rules ? in.rule_off[in.n_states] : 0;
    int n_prev = 0, n_assign = 0, n_valid = 0, rm_active = 0;
    for (int p = 0; p < in.n_parts; ++p) { n_prev += in.part_in_prev[p] != 0; n_assign += in.part_in_assign[p] != 0; }
    for (int q = 0; q < in.n_nodes; ++q) n_valid += in.node_removed[q] == 0;
    for (int q = 0; q < in.n_node_ids; ++q) rm_active |= in.node_removed[q] != 0;
    D.n_assign = n_assign; D.n_valid = n_valid;
    D.P = n_prev; D.rm_active = rm_active; D.add_active = 1; D.add_is_nil = in.add_is_nil; D.use_rest = 0;
    D.active = in.max_iters > 0 ? 1 : 0;
    D.part_off = pl->PT; D.rows_off = pl->RT; D.node_off = pl->NT; D.nodeid_off = pl->NUT;
    D.counts_off = pl->CT; D.n2n_off = pl->N2T; D.mask_off = pl->MT; D.stream_off = pl->ST;
    pl->raw_rows_off[i] = pl->RRT; pl->raw_shape_off[i] = pl->RST;
    seg_off[i] = (int)pl->PT;
    pl->ST += (long long)D.PU * (D.SLP + 8);
    pl->PT += D.PU; pl->RT += (long long)D.PU * D.SLP; pl->NT += D.N; pl->NUT += D.NU;
    pl->CT += (long long)D.S * D.N; pl->N2T += (long long)(D.NU + 1) * D.N;
    pl->MT += (long long)D.n_rules * (D.NU + 1) * D.HW;
    pl->RRT += (long long)D.PU * D.SL; pl->RST += (long long)D.PU * D.S;
    pl->max_N = std::max(pl->max_N, D.N); pl->max_S = std::max(pl->max_S, D.S); pl->max_NU = std::max(pl->max_NU, D.NU);
  }
  seg_off[n] = (int)pl->PT;
  pl->raw_rows_off[n] = pl->RRT; pl->raw_shape_off[n] = pl->RST;
  if (pl->PT >= (1LL << 29)) { plan_release(pl, ctx); return fail(ctx, BLANCE_ERR_UNSUPPORTED, "2^29 or more partitions in one batch"); }
  {
    int top_bits = 1, inst_bits = 1;
    while ((1ll << top_bits) < (long long)pl->max_NU + 2) ++top_bits;
    while ((1ll << inst_bits) < (long long)n + 1) ++inst_bits;
    pl->pair_inst_shift = 13 + top_bits;
    pl->pair_end_bit = pl->pair_inst_shift + inst_bits;
  }

  // ---- carve one device arena ------------------------------------------------------------
  struct Slice { void** ptr; size_t bytes; };
  std::vector<Slice> slices;
  DPool& P = pl->pool;
  const size_t PT = (size_t)pl->PT + 1, RT = (size_t)pl->RT + 4, NT = (size_t)pl->NT + 1, NUT = (size_t)pl->NUT + 1;
  const size_t CT = (size_t)pl->CT + 1, N2T = (size_t)pl->N2T + 1, MT = (size_t)pl->MT + 1;
  const size_t RRT = (size_t)pl->RRT + 1, RST = (size_t)pl->RST + 1;
  const int32_t *c_pweight, *c_rank, *c_inst, *c_nw, *c_ef, *c_er;
  const uint8_t *c_rm, *c_ad, *c_hw;
  const uint32_t* c_mask;
#define SL_(p, T, cnt) slices.push_back(Slice{(void**)&(p), sizeof(T) * (cnt)})
  SL_(P.rows, int32_t, RT); SL_(P.prev_rows, int32_t, RT); SL_(pl->rows_init, int32_t, RT); SL_(pl->prev_rows_init, int32_t, RT);
  SL_(P.pmeta, uint32_t, PT); SL_(P.prev_meta, uint32_t, PT); SL_(pl->pmeta_init, uint32_t, PT); SL_(pl->prev_meta_init, uint32_t, PT);
  SL_(P.pflags, uint8_t, PT); SL_(pl->pflags_init, uint8_t, PT);
  SL_(c_pweight, int32_t, PT); SL_(c_rank, int32_t, PT); SL_(c_inst, int32_t, PT);
  SL_(P.stream, int32_t, (size_t)pl->ST + 4); SL_(P.ostream, int32_t, (size_t)pl->ST + 4);
  SL_(P.keys, unsigned long long, PT); SL_(P.keys_alt, unsigned long long, PT); SL_(P.order, int32_t, PT); SL_(P.order_alt, int32_t, PT);
  SL_(c_rm, uint8_t, NUT); SL_(c_ad, uint8_t, NUT); SL_(c_nw, int32_t, NT); SL_(c_hw, uint8_t, NT);
  SL_(c_ef, int32_t, NT); SL_(c_er, int32_t, NT);
  SL_(P.counts, int32_t, CT); SL_(P.n2n, int32_t, N2T); SL_(c_mask, uint32_t, MT);
  SL_(P.n2n_dev, int32_t, N2T); SL_(P.qstat, int32_t, 4 * PT); SL_(P.srank, uint8_t, PT);
  SL_(P.pair_keys, unsigned long long, 4 * PT); SL_(P.pair_keys_alt, unsigned long long, 4 * PT);
  SL_(P.pair_vals, uint32_t, 4 * PT); SL_(P.pair_vals_alt, uint32_t, 4 * PT);
  SL_(P.insts, DInst, (size_t)n);
  SL_(pl->raw_a, int32_t, RRT); SL_(pl->raw_b, int32_t, RRT); SL_(pl->rawsh_a, uint8_t, RST); SL_(pl->rawsh_b, uint8_t, RST);
  SL_(pl->d_raw_rows_off, long long, (size_t)n + 1); SL_(pl->d_raw_shape_off, long long, (size_t)n + 1);
  SL_(pl->d_seg_off, int, (size_t)n + 1);
#undef SL_
  size_t total = 0;
  for (auto& s : slices) total += align_up(s.bytes, 256);
  // stream-ordered allocation: the context's memory pool keeps the arena of the previous call around
  cudaError_t e = cudaMallocAsync(&pl->arena, total, ctx->stream);
  if (e != cudaSuccess) {
    plan_release(pl, ctx);
    return fail(ctx, BLANCE_ERR_NOMEM, std::string("cudaMalloc of the plan arena failed: ") + cudaGetErrorString(e));
  }
  pl->arena_bytes = total;
  {
    size_t off = 0;
    for (auto& s : slices) { *s.ptr = (char*)pl->arena + off; off += align_up(s.bytes, 256); }
  }
  P.pweight = c_pweight; P.name_rank = c_rank; P.part_inst = c_inst;
  P.node_removed = c_rm; P.node_added = c_ad; P.node_weight = c_nw; P.node_has_weight = c_hw;
  P.extra_first = c_ef; P.extra_rest = c_er; P.ie_mask = c_mask;

  // ---- host side of the copy.  A batch is concatenated in caller layout into one pinned staging buffer;
  // a single instance is copied straight from the caller's arrays (no staging, no pinned allocation).
  const bool direct = (n == 1);
  const int32_t *h_cur = nullptr, *h_prev = nullptr, *h_pw = nullptr, *h_rank = nullptr, *h_inst = nullptr;
  const int32_t *h_nw = nullptr, *h_ef = nullptr, *h_er = nullptr;
  const uint8_t *h_csh = nullptr, *h_psh = nullptr, *h_flags = nullptr, *h_rm = nullptr, *h_ad = nullptr, *h_hw = nullptr;
  const uint32_t* h_mask = nullptr;
  std::vector<uint8_t> v_flags;
  if (direct) {
    const blance_plan_in& in = ins[0];
    const DInst& D = pl->h_insts[0];
    v_flags.resize((size_t)D.PU + 1);
    for (int p = 0; p < D.PU; ++p)
      v_flags[p] = (uint8_t)((in.part_in_prev[p] ? PF_IN_PREV : 0) | ((in.part_in_prev[p] & 2) ? PF_PREV_EXTRA : 0) | (in.part_in_assign[p] ? PF_IN_ASSIGN : 0) |
                             (in.part_has_weight[p] ? PF_HAS_WEIGHT : 0));
    h_cur = in.cur_rows; h_prev = in.prev_rows; h_csh = in.cur_shape; h_psh = in.prev_shape;
    h_flags = v_flags.data(); h_pw = in.part_weight; h_rank = in.part_name_rank;     // h_inst stays NULL: all zero
    h_rm = in.node_removed; h_ad = in.node_added;
    if (in.has_node_weights) { h_nw = in.node_weight; h_hw = in.node_has_weight; }
    h_ef = in.extra_tot_first; h_er = in.extra_tot_rest; h_mask = in.ie_mask;
  } else {
  const size_t stage_bytes = align_up(sizeof(int32_t) * RRT, 256) * 2 + align_up(RST, 256) * 2 + align_up(PT, 256) +
                             align_up(sizeof(int32_t) * PT, 256) * 3 + align_up(NUT, 256) * 2 +
                             align_up(sizeof(int32_t) * NT, 256) * 3 + align_up(NT, 256) + align_up(sizeof(uint32_t) * MT, 256);
  if (stage_bytes > ctx->h_stage_bytes) {          // grow-only, kept by the context between calls
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    ctx->h_stage = nullptr; ctx->h_stage_bytes = 0;
    e = cudaMallocHost(&ctx->h_stage, stage_bytes + stage_bytes / 4);
    if (e != cudaSuccess) {
      plan_release(pl, ctx);
      return fail(ctx, BLANCE_ERR_NOMEM, std::string("cudaMallocHost of the staging buffer failed: ") + cudaGetErrorString(e));
    }
    ctx->h_stage_bytes = stage_bytes + stage_bytes / 4;
  }
  pl->h_stage = ctx->h_stage;
  pl->h_stage_bytes = stage_bytes;
  char* hp = (char*)pl->h_stage;
  auto carve = [&](size_t bytes) { char* r = hp; hp += align_up(bytes, 256); return r; };
  int32_t* s_cur = (int32_t*)carve(sizeof(int32_t) * RRT);
  int32_t* s_prev = (int32_t*)carve(sizeof(int32_t) * RRT);
  uint8_t* s_csh = (uint8_t*)carve(RST);
  uint8_t* s_psh = (uint8_t*)carve(RST);
  uint8_t* s_flags = (uint8_t*)carve(PT);
  int32_t* s_pw = (int32_t*)carve(sizeof(int32_t) * PT);
  int32_t* s_rank = (int32_t*)carve(sizeof(int32_t) * PT);
  int32_t* s_inst = (int32_t*)carve(sizeof(int32_t) * PT);
  uint8_t* s_rm = (uint8_t*)carve(NUT);
  uint8_t* s_ad = (uint8_t*)carve(NUT);
  int32_t* s_nw = (int32_t*)carve(sizeof(int32_t) * NT);
  int32_t* s_ef = (int32_t*)carve(sizeof(int32_t) * NT);
  int32_t* s_er = (int32_t*)carve(sizeof(int32_t) * NT);
  uint8_t* s_hw = (uint8_t*)carve(NT);
  uint32_t* s_mask = (uint32_t*)carve(sizeof(uint32_t) * MT);
  auto stage_one = [&](int i) {
    const blance_plan_in& in = ins[i];
    const DInst& D = pl->h_insts[i];
    const size_t rr = (size_t)D.PU * D.SL, rs = (size_t)D.PU * D.S;
    if (rr) { std::memcpy(s_cur + pl->raw_rows_off[i], in.cur_rows, sizeof(int32_t) * rr);
              std::memcpy(s_prev + pl->raw_rows_off[i], in.prev_rows, sizeof(int32_t) * rr); }
    if (rs) { std::memcpy(s_csh + pl->raw_shape_off[i], in.cur_shape, rs); std::memcpy(s_psh + pl->raw_shape_off[i], in.prev_shape, rs); }
    for (int p = 0; p < D.PU; ++p) {
      const size_t g = (size_t)D.part_off + p;
      s_flags[g] = (uint8_t)((in.part_in_prev[p] ? PF_IN_PREV : 0) | ((in.part_in_prev[p] & 2) ? PF_PREV_EXTRA : 0) | (in.part_in_assign[p] ? PF_IN_ASSIGN : 0) |
                             (in.part_has_weight[p] ? PF_HAS_WEIGHT : 0));
      s_pw[g] = in.part_weight[p];
      s_rank[g] = in.part_name_rank[p];
      s_inst[g] = i;
    }
    if (D.NU) { std::memcpy(s_rm + D.nodeid_off, in.node_removed, D.NU); std::memcpy(s_ad + D.nodeid_off, in.node_added, D.NU); }
    for (int q = 0; q < D.N; ++q) {
      s_nw[D.node_off + q] = in.has_node_weights ? in.node_weight[q] : 0;
      s_hw[D.node_off + q] = in.has_node_weights ? in.node_has_weight[q] : 0;
      s_ef[D.node_off + q] = in.extra_tot_first ? in.extra_tot_first[q] : 0;
      s_er[D.node_off + q] = in.extra_tot_rest ? in.extra_tot_rest[q] : 0;
    }
    const size_t mw = (size_t)D.n_rules * (D.NU + 1) * D.HW;
    if (mw) std::memcpy(s_mask + D.mask_off, in.ie_mask, sizeof(uint32_t) * mw);
  };
  {
    // instances are staged by a few host threads (a 1 024-instance fan-out is ~1 M partitions of flag packing)
    int T = (int)std::min<long long>(8, std::max<long long>(1, pl->PT / 65536));
    T = std::min(T, std::max(1, (int)std::thread::hardware_concurrency()));
    if (T <= 1) { for (int i = 0; i < n; ++i) stage_one(i); }
    else {
      std::vector<std::thread> th;
      for (int t = 0; t < T; ++t) th.emplace_back([&, t]() { for (int i = t; i < n; i += T) stage_one(i); });
      for (auto& x : th) x.join();
    }
  }
  h_cur = s_cur; h_prev = s_prev; h_csh = s_csh; h_psh = s_psh; h_flags = s_flags; h_pw = s_pw; h_rank = s_rank;
  h_inst = s_inst; h_rm = s_rm; h_ad = s_ad; h_nw = s_nw; h_hw = s_hw; h_ef = s_ef; h_er = s_er; h_mask = s_mask;
  }
  cudaStream_t st = ctx->stream;
#define H2D(dst, src, bytes) do { if ((bytes) > 0) { \
    e = (src) ? cudaMemcpyAsync((void*)(dst), (src), (bytes), cudaMemcpyHostToDevice, st) : cudaMemsetAsync((void*)(dst), 0, (bytes), st); \
    if (e != cudaSuccess) { plan_release(pl, ctx); return fail(ctx, BLANCE_ERR_CUDA, std::string("H2D copy failed: ") + cudaGetErrorString(e)); } } } while (0)
  H2D(pl->raw_a, h_cur, sizeof(int32_t) * (size_t)pl->RRT); H2D(pl->raw_b, h_prev, sizeof(int32_t) * (size_t)pl->RRT);
  H2D(pl->rawsh_a, h_csh, (size_t)pl->RST); H2D(pl->rawsh_b, h_psh, (size_t)pl->RST);
  H2D(pl->pflags_init, h_flags, (size_t)pl->PT); H2D(c_pweight, h_pw, sizeof(int32_t) * (size_t)pl->PT);
  H2D(c_rank, h_rank, sizeof(int32_t) * (size_t)pl->PT); H2D(c_inst, h_inst, sizeof(int32_t) * (size_t)pl->PT);
  H2D(c_rm, h_rm, (size_t)pl->NUT); H2D(c_ad, h_ad, (size_t)pl->NUT);
  H2D(c_nw, h_nw, sizeof(int32_t) * (size_t)pl->NT); H2D(c_hw, h_hw, (size_t)pl->NT);
  H2D(c_ef, h_ef, sizeof(int32_t) * (size_t)pl->NT); H2D(c_er, h_er, sizeof(int32_t) * (size_t)pl->NT);
  H2D(c_mask, h_mask, sizeof(uint32_t) * (size_t)pl->MT);
  H2D(P.insts, pl->h_insts.data(), sizeof(DInst) * (size_t)n);
  H2D(pl->d_raw_rows_off, pl->raw_rows_off.data(), sizeof(long long) * (size_t)(n + 1));
  H2D(pl->d_raw_shape_off, pl->raw_shape_off.data(), sizeof(long long) * (size_t)(n + 1));
  H2D(pl->d_seg_off, seg_off.data(), sizeof(int) * (size_t)(n + 1));
#undef H2D
  // device layout of the rows / shapes, into the *_init copies via the working arrays
  if (pl->PT > 0) {
    k_unpack<<<grid_for(ctx, pl->PT, 256), 256, 0, st>>>(P, pl->raw_a, pl->raw_b, pl->rawsh_a, pl->rawsh_b,
                                                        pl->d_raw_rows_off, pl->d_raw_shape_off, pl->PT);
    ctx->launches++;
    e = cudaGetLastError();
    if (e != cudaSuccess) { plan_release(pl, ctx); return fail(ctx, BLANCE_ERR_CUDA, std::string("k_unpack launch failed: ") + cudaGetErrorString(e)); }
    if (e == cudaSuccess) e = cudaMemcpyAsync(pl->rows_init, P.rows, sizeof(int32_t) * (size_t)pl->RT, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(pl->prev_rows_init, P.prev_rows, sizeof(int32_t) * (size_t)pl->RT, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(pl->pmeta_init, P.pmeta, sizeof(uint32_t) * (size_t)pl->PT, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(pl->prev_meta_init, P.prev_meta, sizeof(uint32_t) * (size_t)pl->PT, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) { plan_release(pl, ctx); return fail(ctx, BLANCE_ERR_CUDA, std::string("upload failed: ") + cudaGetErrorString(e)); }
  }
  // sort scratch
  size_t need = 0, need2 = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, need, P.keys_alt, P.keys, P.order_alt, P.order, (int)pl->PT, 0, 64, st);
  cub::DeviceSegmentedRadixSort::SortPairs(nullptr, need2, P.keys_alt, P.keys, P.order_alt, P.order, (int)pl->PT, n,
                                           pl->d_seg_off, pl->d_seg_off + 1, 0, 64, st);
  need = std::max(need, need2);
  {
    size_t need3 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, need3, P.pair_keys_alt, P.pair_keys, P.pair_vals_alt, P.pair_vals, (int)(4 * pl->PT), 0, 64, st);
    need = std::max(need, need3);
  }
  if (need > ctx->cub_tmp_bytes) {
    if (ctx->cub_tmp) cudaFree(ctx->cub_tmp);
    ctx->cub_tmp = nullptr; ctx->cub_tmp_bytes = 0;
    e = cudaMalloc(&ctx->cub_tmp, need);
    if (e != cudaSuccess) { plan_release(pl, ctx); return fail(ctx, BLANCE_ERR_NOMEM, "cudaMalloc of the sort scratch failed"); }
    ctx->cub_tmp_bytes = need;
  }
  e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) { plan_release(pl, ctx); return fail(ctx, BLANCE_ERR_CUDA, std::string("upload sync failed: ") + cudaGetErrorString(e)); }
  *out_plan = pl;
  return BLANCE_OK;
}

static cudaEvent_t get_event(blance_ctx* ctx, size_t idx) {
  while (ctx->events.size() <= idx) {
    cudaEvent_t ev;
    if (cudaEventCreate(&ev) != cudaSuccess) return nullptr;
    ctx->events.push_back(ev);
  }
  return ctx->events[idx];
}

template <int NPT, int MAXT>
static void launch_pass(const DPool& P, int n_inst, int T, int s, bool hier, cudaStream_t st) {
  if (hier) k_assign_pass<NPT, true, MAXT><<<n_inst, T, 0, st>>>(P, s);
  else k_assign_pass<NPT, false, MAXT><<<n_inst, T, 0, st>>>(P, s);
}

// the sequencer variant, one instantiation per constraint count K; CTAs whose instance picked the other
// kernel (or has a different K for this state) exit at once
template <int NPT, int K, int MAXT>
static cudaError_t launch_pass_seq_k(size_t* configured, const DPool& P, int n_inst, int TC, int W, int s, size_t dyn, cudaStream_t st) {
  {
    std::lock_guard<std::mutex> g(g_seq_dyn_mu);
    if (dyn > *configured) {
      cudaError_t e = cudaFuncSetAttribute(k_assign_pass_seq<NPT, K, MAXT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      if (e != cudaSuccess) return e;
      *configured = dyn;
    }
  }
  k_assign_pass_seq<NPT, K, MAXT><<<n_inst, TC + 32 * W, dyn, st>>>(P, s, TC);
  return cudaSuccess;
}

// kmask: bit K set when some instance of the batch has constraints == K for state s
template <int NPT, int MAXT>
static cudaError_t launch_pass_seq(size_t* configured, const DPool& P, int n_inst, int TC, int W, int s, int max_n, unsigned kmask, cudaStream_t st) {
  const size_t dyn = seq_dyn_smem_bytes(max_n, W);
  cudaError_t e = cudaSuccess;
  if (e == cudaSuccess && (kmask & 2u)) e = launch_pass_seq_k<NPT, 1, MAXT>(configured + 0, P, n_inst, TC, W, s, dyn, st);
  if (e == cudaSuccess && (kmask & 4u)) e = launch_pass_seq_k<NPT, 2, MAXT>(configured + 1, P, n_inst, TC, W, s, dyn, st);
  if (e == cudaSuccess && (kmask & 8u)) e = launch_pass_seq_k<NPT, 3, MAXT>(configured + 2, P, n_inst, TC, W, s, dyn, st);
  if (e == cudaSuccess && (kmask & 16u)) e = launch_pass_seq_k<NPT, 4, MAXT>(configured + 3, P, n_inst, TC, W, s, dyn, st);
  return e;
}

// the speculative variant, one instantiation per constraint count K (CTAs of other modes / other K exit at once)
template <int K>
static cudaError_t launch_pass_spec_k(size_t* configured, const DPool& P, int n_inst, int nw, int sw, unsigned idle_mask, int shift, int s, size_t dyn, cudaStream_t st) {
  {
    std::lock_guard<std::mutex> g(g_seq_dyn_mu);
    if (dyn > *configured) {
      cudaError_t e = cudaFuncSetAttribute(k_assign_pass_spec<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      if (e != cudaSuccess) return e;
      *configured = dyn;
    }
  }
  k_assign_pass_spec<K><<<n_inst, 32 * nw, dyn, st>>>(P, s, sw, idle_mask, shift);
  return cudaSuccess;
}

static int next_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }

// Compute threads per CTA (TC, a power of two; the kernel adds one service warp) and nodes per
// thread for the pass kernel.  The chain is latency bound, so prefer many warps with few nodes each.
static void pass_shape(int max_n, int* TC, int* npt) {
  int want = max_n > 512 ? 2 : 1;
  if (const char* e = getenv("BLANCE_PASS_NPT")) { int v = atoi(e); if (v == 1 || v == 2 || v == 4 || v == 8) want = v; }
  if (max_n > 3968) want = 8;
  int t = next_pow2((std::max(1, max_n) + want - 1) / want);
  if (t < 32) t = 32;
  if (t > 512) t = 512;
  int n = (max_n + t - 1) / t;
  *npt = n <= 1 ? 1 : n <= 2 ? 2 : n <= 4 ? 4 : n <= 8 ? 8 : 16;
  *TC = t;
}

static int run(blance_ctx* ctx, blance_plan* pl) {
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  DPool& P = pl->pool;
  const int n = pl->n_inst;
  // restore the mutable state
  if (pl->PT > 0) {
    CK(cudaMemcpyAsync(P.rows, pl->rows_init, sizeof(int32_t) * (size_t)pl->RT, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(P.prev_rows, pl->prev_rows_init, sizeof(int32_t) * (size_t)pl->RT, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(P.pmeta, pl->pmeta_init, sizeof(uint32_t) * (size_t)pl->PT, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(P.prev_meta, pl->prev_meta_init, sizeof(uint32_t) * (size_t)pl->PT, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(P.pflags, pl->pflags_init, (size_t)pl->PT, cudaMemcpyDeviceToDevice, st));
  }
  CK(cudaMemcpyAsync(P.insts, pl->h_insts.data(), sizeof(DInst) * (size_t)n, cudaMemcpyHostToDevice, st));
  CK(cudaEventRecord(ctx->ev[1], st));

  int T = 32, npt = 1;
  pass_shape(pl->max_N, &T, &npt);
  bool any_hier = false;
  for (int i = 0; i < n; ++i) any_hier |= pl->h_insts[i].has_hier_rules != 0;
  int any_active = 0;
  for (int i = 0; i < n; ++i) any_active += pl->h_insts[i].active;
  const int blk = 256;
  const int grid = grid_for(ctx, pl->PT, blk);
  size_t n_ev = 0;
  pl->pass_launches = 0;
  const bool smem_hist = (n == 1) && ((size_t)pl->h_insts[0].S * pl->h_insts[0].N * sizeof(int32_t) <= 40 * 1024);
  int guard = 0;
  while (any_active > 0) {
    if (++guard > 100000) return fail(ctx, BLANCE_ERR_CUDA, "convergence loop did not terminate");
    if (pl->PT == 0) {          // no partitions at all: the loop of plan.go:32-45 still runs once and matches
      CK(cudaMemsetAsync(ctx->d_any_active, 0, sizeof(int), st));
      k_next_iter<<<(n + 127) / 128, 128, 0, st>>>(P, n, ctx->d_any_active);
      ctx->launches++;
      break;
    }
    k_prepare_rows<<<grid, blk, 0, st>>>(P, pl->PT);
    ctx->launches += 2;   // + k_count_prev below
    CK(cudaMemsetAsync(P.counts, 0, sizeof(int32_t) * (size_t)(pl->CT + 1), st));
    if (smem_hist)
      k_count_prev<true><<<std::min(grid, ctx->sm_count * 2), blk, (size_t)pl->h_insts[0].S * pl->h_insts[0].N * sizeof(int32_t), st>>>(P, pl->PT);
    else
      k_count_prev<false><<<grid, blk, 0, st>>>(P, pl->PT);
    for (int s = 0; s < pl->max_S; ++s) {
      if (!pl->any_state_active[s]) continue;
      k_build_keys<<<grid, blk, 0, st>>>(P, s, pl->PT);
      ctx->launches += 2;   // + k_assign_pass below
      size_t tmp = ctx->cub_tmp_bytes;
      if (n == 1)
        CK(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp, tmp, P.keys_alt, P.keys, P.order_alt, P.order, (int)pl->PT, 0, 64, st));
      else
        CK(cub::DeviceSegmentedRadixSort::SortPairs(ctx->cub_tmp, tmp, P.keys_alt, P.keys, P.order_alt, P.order, (int)pl->PT,
                                                    n, pl->d_seg_off, pl->d_seg_off + 1, 0, 64, st));
      k_gather_stream<<<grid, blk, 0, st>>>(P, s, pl->PT);
      unsigned kmask = 0;
      for (int i = 0; i < n; ++i) { const int kk = pl->h_insts[i].S > s ? pl->h_insts[i].state_constraints[s] : 0; if (kk >= 1 && kk <= 4) kmask |= 1u << kk; }
      // speculative kernel: 9 scout warps + the leader (warps 4 and 8 stay away from the leader's scheduler) when the
      // GPU has SMs to spare, 3 scouts per CTA for wide batches
      // speculative kernel: warp 0 leads, 9 scout warps (warps 4 and 8 exit at once: the leader has its scheduler to
      // itself) when the GPU has SMs to spare; leader + 3 scouts per CTA for wide batches
      const bool spec_wide = 2 * n <= ctx->sm_count;
      const int spec_nw = spec_wide ? 12 : 4, spec_sw = spec_wide ? 9 : 3;
      const unsigned spec_idle = spec_wide ? ((1u << 4) | (1u << 8)) : 0u;
      const int spec_shift = 0;
      const int spec_max_n = std::min(2048, 32 * spec_sw * SP_NPTS);
      bool any_auto = false;
      for (int i = 0; i < n; ++i) any_auto |= pl->h_insts[i].engine == BLANCE_ENGINE_AUTO;
      const bool spec_allowed = any_auto && kmask != 0 && pl->pair_end_bit <= 62 && !getenv("BLANCE_NO_SPEC");
      k_pick_mode<<<(n + 127) / 128, 128, 0, st>>>(P, s, n, (npt <= 8 && !getenv("BLANCE_NO_SEQ")) ? 1 : 0, spec_allowed ? 1 : 0, spec_max_n);
      if (spec_allowed) {
        // the all-sticky hypothesis counts (qstat) of the instances that picked the speculative kernel
        k_pair_keys<<<grid, blk, 0, st>>>(P, s, pl->PT, pl->pair_inst_shift);
        size_t tmp2 = ctx->cub_tmp_bytes;
        CK(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp, tmp2, P.pair_keys_alt, P.pair_keys, P.pair_vals_alt, P.pair_vals,
                                           (int)(4 * pl->PT), 0, pl->pair_end_bit + 1, st));
        k_pair_rank<<<grid_for(ctx, 4 * pl->PT, blk), blk, 0, st>>>(P, 4 * pl->PT);
        CK(cudaMemsetAsync(P.n2n_dev, 0, sizeof(int32_t) * (size_t)(pl->N2T + 1), st));
        ctx->launches += 2;
      }
      CK(cudaMemsetAsync(P.n2n, 0, sizeof(int32_t) * (size_t)(pl->N2T + 1), st));     // plan.go:266
      cudaEvent_t e0 = get_event(ctx, n_ev), e1 = get_event(ctx, n_ev + 1);
      if (e0 && e1 && n_ev < 256) CK(cudaEventRecord(e0, st));
      if (npt == 1) launch_pass<1, 544>(P, n, T + 32, s, any_hier, st);
      else if (npt == 2) launch_pass<2, 544>(P, n, T + 32, s, any_hier, st);
      else if (npt == 4) launch_pass<4, 544>(P, n, T + 32, s, any_hier, st);
      else if (npt == 8) launch_pass<8, 544>(P, n, T + 32, s, any_hier, st);
      else launch_pass<16, 544>(P, n, T + 32, s, any_hier, st);
      cudaError_t se = cudaSuccess;
      // sequencer warps per CTA: wide windows when the GPU has SMs to spare, one warp for wide batches
      int seq_w = (2 * n <= ctx->sm_count) ? SEQ_W_MAX : 1;
      if (const char* ev = getenv("BLANCE_SEQ_W")) { const int v = atoi(ev); if (v >= 1 && v <= SEQ_W_MAX) seq_w = v; }   // experiments
      if (npt == 1) se = (launch_pass_seq<1, 640>)(g_seq_dyn[ctx->device & 63][0], P, n, T, seq_w, s, pl->max_N, kmask, st);
      else if (npt == 2) se = (launch_pass_seq<2, 640>)(g_seq_dyn[ctx->device & 63][1], P, n, T, seq_w, s, pl->max_N, kmask, st);
      else if (npt == 4) se = (launch_pass_seq<4, 640>)(g_seq_dyn[ctx->device & 63][2], P, n, T, seq_w, s, pl->max_N, kmask, st);
      else if (npt == 8) se = (launch_pass_seq<8, 640>)(g_seq_dyn[ctx->device & 63][3], P, n, T, seq_w, s, pl->max_N, kmask, st);
      CK(se);
      CK(cudaGetLastError());
      ctx->launches += 1 + (npt <= 8 ? __builtin_popcount(kmask) : 0);   // k_pick_mode + the sequencer kernel(s)
      if (spec_allowed) {
        const size_t sdyn = spec_dyn_smem_bytes(std::min(pl->max_N, spec_max_n), spec_sw);
        size_t* cfgd = g_spec_dyn[ctx->device & 63];
        cudaError_t pe = cudaSuccess;
        if (pe == cudaSuccess && (kmask & 2u)) pe = launch_pass_spec_k<1>(cfgd + 0, P, n, spec_nw, spec_sw, spec_idle, spec_shift, s, sdyn, st);
        if (pe == cudaSuccess && (kmask & 4u)) pe = launch_pass_spec_k<2>(cfgd + 1, P, n, spec_nw, spec_sw, spec_idle, spec_shift, s, sdyn, st);
        if (pe == cudaSuccess && (kmask & 8u)) pe = launch_pass_spec_k<3>(cfgd + 2, P, n, spec_nw, spec_sw, spec_idle, spec_shift, s, sdyn, st);
        if (pe == cudaSuccess && (kmask & 16u)) pe = launch_pass_spec_k<4>(cfgd + 3, P, n, spec_nw, spec_sw, spec_idle, spec_shift, s, sdyn, st);
        CK(pe);
        ctx->launches += __builtin_popcount(kmask);
      }
      CK(cudaGetLastError());
      if (e0 && e1 && n_ev < 256) { CK(cudaEventRecord(e1, st)); n_ev += 2; }
      pl->pass_launches++;
      k_scatter_stream<<<grid, blk, 0, st>>>(P, s, pl->PT);
      ctx->launches += 2;   // gather + scatter
    }
    k_compare<<<grid, blk, 0, st>>>(P, pl->PT);
    ctx->launches += 3;   // + k_commit, k_next_iter
    k_commit<<<grid, blk, 0, st>>>(P, pl->PT);
    CK(cudaMemsetAsync(ctx->d_any_active, 0, sizeof(int), st));
    k_next_iter<<<(n + 127) / 128, 128, 0, st>>>(P, n, ctx->d_any_active);
    CK(cudaMemcpyAsync(ctx->h_any_active, ctx->d_any_active, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    any_active = *ctx->h_any_active;
  }
  CK(cudaEventRecord(ctx->ev[2], st));
  CK(cudaStreamSynchronize(st));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, ctx->ev[1], ctx->ev[2]));
  pl->last_kernel_ms = ms;
  float pass = 0.f;
  const bool show = getenv("BLANCE_PASS_TIMES") != nullptr;
  for (size_t i = 0; i + 1 < n_ev; i += 2) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, ctx->events[i], ctx->events[i + 1]) == cudaSuccess) pass += t;
    if (show) std::fprintf(stderr, "[blance] assign pass %zu: %.3f ms\n", i / 2, t);
  }
  pl->last_pass_ms = pass;
  return BLANCE_OK;
}

static int fetch(blance_ctx* ctx, blance_plan* pl, blance_plan_out* outs) {
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int n = pl->n_inst;
  if (pl->PT > 0) {
    k_pack<<<grid_for(ctx, pl->PT, 256), 256, 0, st>>>(pl->pool, pl->raw_a, pl->rawsh_a, pl->rawsh_b, pl->d_raw_rows_off,
                                                      pl->d_raw_shape_off, pl->PT);
    CK(cudaGetLastError());
    ctx->launches++;
  }
  // a single instance is copied straight into the caller's buffers; a batch lands in the pinned staging
  // buffer first (its head is large enough: it held cur+prev rows)
  int32_t* h_rows = nullptr;
  uint8_t *h_shape = nullptr, *h_warn = nullptr;
  const bool direct = pl->h_stage == nullptr;
  if (direct) {
    h_rows = outs[0].next_rows; h_shape = outs[0].next_shape; h_warn = outs[0].warn;
  } else {
    char* hp = (char*)pl->h_stage;
    h_rows = (int32_t*)hp;
    hp += align_up(sizeof(int32_t) * ((size_t)pl->RRT + 1), 256) * 2;
    h_shape = (uint8_t*)hp;
    hp += align_up((size_t)pl->RST + 1, 256);
    h_warn = (uint8_t*)hp;
  }
  if (pl->RRT && h_rows) CK(cudaMemcpyAsync(h_rows, pl->raw_a, sizeof(int32_t) * (size_t)pl->RRT, cudaMemcpyDeviceToHost, st));
  if (pl->RST && h_shape) CK(cudaMemcpyAsync(h_shape, pl->rawsh_a, (size_t)pl->RST, cudaMemcpyDeviceToHost, st));
  if (pl->RST && h_warn) CK(cudaMemcpyAsync(h_warn, pl->rawsh_b, (size_t)pl->RST, cudaMemcpyDeviceToHost, st));
  std::vector<DInst> fin(n);
  CK(cudaMemcpyAsync(fin.data(), pl->pool.insts, sizeof(DInst) * (size_t)n, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (int i = 0; i < n; ++i)
    if (fin[i].spec_abort) return fail(ctx, BLANCE_ERR_CUDA, "the speculative pass kernel gave up waiting (internal error; see stderr of the device printf)");
  if (getenv("BLANCE_SPEC_STATS"))
    for (int i = 0; i < n && i < 4; ++i)
      std::fprintf(stderr, "[blance] inst %d: steps %lld accepted %lld | resolved by the leader %lld (stale results %lld) movers %lld team %lld rebuilds %lld waits %lld\n",
                   i, fin[i].steps, fin[i].fast_steps, fin[i].spec_resolved, fin[i].spec_stale, fin[i].spec_movers, fin[i].spec_team,
                   fin[i].spec_rebuilds, fin[i].spec_waits),
      std::fprintf(stderr, "[blance]   leader cycles (-DBLANCE_SPEC_TIMING builds): scans %lld | waits %lld | resolves %lld | mover updates %lld | team %lld | passes total %lld\n",
                   fin[i].spec_cyc[0], fin[i].spec_cyc[1], fin[i].spec_cyc[2], fin[i].spec_cyc[3], fin[i].spec_cyc[4], fin[i].spec_cyc[5]);
  for (int i = 0; i < n; ++i) {
    const DInst& D = pl->h_insts[i];
    blance_plan_out& o = outs[i];
    const size_t rr = (size_t)D.PU * D.SL, rs = (size_t)D.PU * D.S;
    if (!direct) {
      if (rr && o.next_rows) std::memcpy(o.next_rows, h_rows + pl->raw_rows_off[i], sizeof(int32_t) * rr);
      if (rs && o.next_shape) std::memcpy(o.next_shape, h_shape + pl->raw_shape_off[i], rs);
      if (rs && o.warn) std::memcpy(o.warn, h_warn + pl->raw_shape_off[i], rs);
    }
    o.iters_run = fin[i].iters_run;
    o.converged = fin[i].converged;
    o.steps = fin[i].steps;
    o.sticky_steps = fin[i].fast_steps;
    o.kernel_ms = pl->last_kernel_ms;
    o.pass_ms = pl->last_pass_ms;
    o.device_ms = 0.f;
  }
  return BLANCE_OK;
}

extern "C" int blance_plan_upload(blance_ctx* ctx, const blance_plan_in* in, blance_plan** plan) {
  if (ctx && !ctx->children.empty()) ctx = ctx->children[0];
  if (!ctx) return fail(nullptr, BLANCE_ERR_INVALID_ARG, "ctx is NULL");
  if (!plan) return fail(ctx, BLANCE_ERR_INVALID_ARG, "plan is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  return upload(ctx, 1, in, plan);
}

extern "C" int blance_plan_run(blance_ctx* ctx, blance_plan* plan) {
  if (ctx && !ctx->children.empty()) ctx = ctx->children[0];
  if (!ctx || !plan) return fail(ctx, BLANCE_ERR_INVALID_ARG, "ctx or plan is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  return run(ctx, plan);
}

extern "C" int blance_plan_fetch(blance_ctx* ctx, blance_plan* plan, blance_plan_out* out) {
  if (ctx && !ctx->children.empty()) ctx = ctx->children[0];
  if (!ctx || !plan || !out) return fail(ctx, BLANCE_ERR_INVALID_ARG, "ctx, plan or out is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  return fetch(ctx, plan, out);
}

extern "C" int blance_plan_timing(const blance_plan* plan, float* kernel_ms, float* pass_ms, int32_t* pass_launches) {
  if (!plan) return BLANCE_ERR_INVALID_ARG;
  if (kernel_ms) *kernel_ms = plan->last_kernel_ms;
  if (pass_ms) *pass_ms = plan->last_pass_ms;
  if (pass_launches) *pass_launches = plan->pass_launches;
  return BLANCE_OK;
}

extern "C" void blance_plan_free(blance_ctx* ctx, blance_plan* plan) {
  if (!plan) return;
  if (ctx && !ctx->children.empty()) ctx = ctx->children[0];
  if (ctx) { std::lock_guard<std::mutex> g(ctx->mu); cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream); plan_release(plan, ctx); }
  else plan_release(plan);
}

static int plan_batch_one(blance_ctx* ctx, int32_t n, const blance_plan_in* in, blance_plan_out* out) {
  std::lock_guard<std::mutex> g(ctx->mu);
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventRecord(ctx->ev[0], ctx->stream));
  blance_plan* pl = nullptr;
  int st = upload(ctx, n, in, &pl);
  if (st != BLANCE_OK) return st;
  st = run(ctx, pl);
  if (st == BLANCE_OK) st = fetch(ctx, pl, out);
  if (st == BLANCE_OK) {
    cudaEventRecord(ctx->ev[3], ctx->stream);
    cudaEventSynchronize(ctx->ev[3]);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[3]);
    for (int i = 0; i < n; ++i) out[i].device_ms = ms;
  }
  plan_release(pl, ctx);
  return st;
}

static int plan_batch(blance_ctx* ctx, int32_t n, const blance_plan_in* in, blance_plan_out* out) {
  if (!ctx) return fail(nullptr, BLANCE_ERR_INVALID_ARG, "ctx is NULL");
  if (!in || !out) return fail(ctx, BLANCE_ERR_INVALID_ARG, "in or out is NULL");
  if (ctx->children.empty()) return plan_batch_one(ctx, n, in, out);
  if (n <= 0) return fail(ctx, BLANCE_ERR_INVALID_ARG, "batch size must be positive");
  // ---- several GPUs: instance i -> device i mod G, one host thread per device, no collective -------------------
  const int G = (int)std::min<size_t>(ctx->children.size(), (size_t)n);
  if (G == 1) {
    const int st = plan_batch_one(ctx->children[0], n, in, out);
    if (st != BLANCE_OK) ctx->err = ctx->children[0]->err;
    return st;
  }
  std::vector<std::vector<blance_plan_in>> ins((size_t)G);
  std::vector<std::vector<blance_plan_out>> outs((size_t)G);
  for (int i = 0; i < n; ++i) { ins[(size_t)(i % G)].push_back(in[i]); outs[(size_t)(i % G)].push_back(out[i]); }
  std::vector<int> status((size_t)G, BLANCE_OK);
  std::vector<std::thread> th;
  for (int d = 0; d < G; ++d)
    th.emplace_back([&, d]() {
      status[(size_t)d] = plan_batch_one(ctx->children[(size_t)d], (int32_t)ins[(size_t)d].size(), ins[(size_t)d].data(), outs[(size_t)d].data());
    });
  for (auto& t : th) t.join();
  for (int d = 0; d < G; ++d)
    if (status[(size_t)d] != BLANCE_OK) {
      ctx->err = "device " + std::to_string(ctx->children[(size_t)d]->device) + ": " + ctx->children[(size_t)d]->err;
      return status[(size_t)d];
    }
  for (int i = 0; i < n; ++i) out[i] = outs[(size_t)(i % G)][(size_t)(i / G)];
  return BLANCE_OK;
}

extern "C" int blance_plan_next_map(blance_ctx* ctx, const blance_plan_in* in, blance_plan_out* out) {
  return plan_batch(ctx, 1, in, out);
}

extern "C" int blance_plan_next_map_batch(blance_ctx* ctx, int32_t n, const blance_plan_in* in, blance_plan_out* out) {
  return plan_batch(ctx, n, in, out);
}

extern "C" int blance_calc_partition_moves(blance_ctx* ctx, int32_t n_parts, int32_t n_states, int32_t n_visit_states,
                                           const int32_t* state_slot_off, const int32_t* beg_rows,
                                           const int32_t* end_rows, int32_t favor_min_nodes, int32_t max_ops,
                                           int32_t* op_node, uint8_t* op_state, uint8_t* op_kind, int32_t* op_count) {
  if (!ctx) return fail(nullptr, BLANCE_ERR_INVALID_ARG, "ctx is NULL");
  if (!ctx->children.empty()) {
    blance_ctx* c0 = ctx->children[0];
    const int st = blance_calc_partition_moves(c0, n_parts, n_states, n_visit_states, state_slot_off, beg_rows, end_rows,
                                               favor_min_nodes, max_ops, op_node, op_state, op_kind, op_count);
    if (st != BLANCE_OK) ctx->err = c0->err;
    return st;
  }
  if (n_parts < 0 || n_states < 0 || n_states >= 255 || n_visit_states < 0 || n_visit_states > n_states || !state_slot_off || max_ops < 0)
    return fail(ctx, BLANCE_ERR_INVALID_ARG, "blance_calc_partition_moves: bad sizes (at most 254 states: 0xFF is the \"\" state of a del op)");
  if (max_ops < 2 * state_slot_off[n_states])
    return fail(ctx, BLANCE_ERR_INVALID_ARG, "blance_calc_partition_moves: max_ops must be at least 2 * n_slots (no op may be dropped)");
  if (n_parts == 0) return BLANCE_OK;
  const int SL = state_slot_off[n_states];
  if (SL > 0 && (!beg_rows || !end_rows)) return fail(ctx, BLANCE_ERR_INVALID_ARG, "rows are NULL");
  if (!op_node || !op_state || !op_kind || !op_count) return fail(ctx, BLANCE_ERR_INVALID_ARG, "outputs are NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t rows_b = sizeof(int32_t) * (size_t)n_parts * std::max(SL, 1), ops = (size_t)n_parts * std::max(max_ops, 1);
  char* d = nullptr;
  const size_t o_slot = 0, o_beg = align_up(sizeof(int32_t) * (n_states + 1), 256), o_end = o_beg + align_up(rows_b, 256),
               o_node = o_end + align_up(rows_b, 256), o_state = o_node + align_up(sizeof(int32_t) * ops, 256),
               o_kind = o_state + align_up(ops, 256), o_cnt = o_kind + align_up(ops, 256),
               total = o_cnt + align_up(sizeof(int32_t) * (size_t)n_parts, 256);
  if (cudaMallocAsync((void**)&d, total, st) != cudaSuccess)       // stream-ordered pool: no device-wide sync per call
    return fail(ctx, BLANCE_ERR_NOMEM, "blance_calc_partition_moves: device allocation failed");
  int rc = BLANCE_OK;
  auto step = [&](cudaError_t e, const char* what) {
    if (e != cudaSuccess && rc == BLANCE_OK) rc = fail(ctx, BLANCE_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  };
  step(cudaMemcpyAsync(d + o_slot, state_slot_off, sizeof(int32_t) * (n_states + 1), cudaMemcpyHostToDevice, st), "H2D");
  if (SL > 0) {
    step(cudaMemcpyAsync(d + o_beg, beg_rows, sizeof(int32_t) * (size_t)n_parts * SL, cudaMemcpyHostToDevice, st), "H2D");
    step(cudaMemcpyAsync(d + o_end, end_rows, sizeof(int32_t) * (size_t)n_parts * SL, cudaMemcpyHostToDevice, st), "H2D");
  }
  if (rc == BLANCE_OK) {
    k_calc_moves<<<grid_for(ctx, n_parts, 128), 128, 0, st>>>(n_parts, n_states, n_visit_states, (const int32_t*)(d + o_slot),
                                                             (const int32_t*)(d + o_beg), (const int32_t*)(d + o_end),
                                                             favor_min_nodes, max_ops, (int32_t*)(d + o_node),
                                                             (uint8_t*)(d + o_state), (uint8_t*)(d + o_kind), (int32_t*)(d + o_cnt));
    step(cudaGetLastError(), "k_calc_moves");
    ctx->launches++;
  }
  if (max_ops > 0) {
    step(cudaMemcpyAsync(op_node, d + o_node, sizeof(int32_t) * (size_t)n_parts * max_ops, cudaMemcpyDeviceToHost, st), "D2H");
    step(cudaMemcpyAsync(op_state, d + o_state, (size_t)n_parts * max_ops, cudaMemcpyDeviceToHost, st), "D2H");
    step(cudaMemcpyAsync(op_kind, d + o_kind, (size_t)n_parts * max_ops, cudaMemcpyDeviceToHost, st), "D2H");
  }
  step(cudaMemcpyAsync(op_count, d + o_cnt, sizeof(int32_t) * (size_t)n_parts, cudaMemcpyDeviceToHost, st), "D2H");
  cudaFreeAsync(d, st);
  step(cudaStreamSynchronize(st), "sync");
  return rc;
}

// ---------------------------------------------------------------------------------------
// Move lists for the orchestrator (orchestrate.go:273-287, 749-763, 177-186), resident on the device.

struct blance_moves {
  int32_t n_parts = 0, n_node_ids = 0;
  long long total_ops = 0;
  char* arena = nullptr;             // one stream-ordered allocation
  long long* d_off = nullptr;        // [n_parts + 1]
  int32_t* d_node = nullptr; uint8_t* d_state = nullptr; uint8_t* d_kind = nullptr;   // CSR ops
  int32_t* d_next = nullptr;         // [n_parts] cursors of the current round
  uint32_t *d_key = nullptr, *d_key2 = nullptr; int32_t *d_val = nullptr, *d_val2 = nullptr;   // [n_parts]
  int32_t* d_ncnt = nullptr; int32_t* d_noff = nullptr; unsigned long long* d_nbest = nullptr; int32_t* d_best = nullptr;   // per node
  void* d_tmp = nullptr; size_t tmp_bytes = 0;
};

extern "C" int blance_moves_create(blance_ctx* ctx, int32_t n_parts, int32_t n_states, int32_t n_visit_states,
                                   const int32_t* state_slot_off, const int32_t* beg_rows, const int32_t* end_rows,
                                   int32_t favor_min_nodes, int32_t n_node_ids, blance_moves** out, int64_t* total_ops) {
  if (!ctx) return fail(nullptr, BLANCE_ERR_INVALID_ARG, "ctx is NULL");
  if (!ctx->children.empty()) ctx = ctx->children[0];
  if (!out) return fail(ctx, BLANCE_ERR_INVALID_ARG, "blance_moves_create: out is NULL");
  *out = nullptr;
  if (n_parts < 0 || n_states < 0 || n_states >= 255 || n_visit_states < 0 || n_visit_states > n_states || !state_slot_off || n_node_ids < 0)
    return fail(ctx, BLANCE_ERR_INVALID_ARG, "blance_moves_create: bad sizes");
  const int SL = state_slot_off[n_states];
  if (n_parts > 0 && SL > 0 && (!beg_rows || !end_rows)) return fail(ctx, BLANCE_ERR_INVALID_ARG, "rows are NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int max_ops = std::max(1, 2 * SL);
  const size_t P = (size_t)std::max(n_parts, 1), NN = (size_t)std::max(n_node_ids, 1);
  // one temp buffer serves the scan of the op counts here, and the sort over partitions and the scan of the
  // n_node_ids + 1 per-node counters in blance_moves_available
  size_t scan_tmp = 0, sort_tmp = 0, node_scan_tmp = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, scan_tmp, (const int32_t*)nullptr, (long long*)nullptr, n_parts + 1, st);
  cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const int32_t*)nullptr, (int32_t*)nullptr, n_parts, 0, 32, st);
  cub::DeviceScan::ExclusiveSum(nullptr, node_scan_tmp, (const int32_t*)nullptr, (int32_t*)nullptr, n_node_ids + 1, st);
  // scratch of the construction (rows, padded ops, counts) lives in the same arena and is simply left unused later
  struct Sl { void** p; size_t bytes; };
  blance_moves* mv = new blance_moves();
  mv->n_parts = n_parts; mv->n_node_ids = n_node_ids;
  int32_t *d_slot = nullptr, *d_beg = nullptr, *d_end = nullptr, *p_node = nullptr, *d_cnt = nullptr;
  uint8_t *p_state = nullptr, *p_kind = nullptr;
  mv->tmp_bytes = std::max({scan_tmp, sort_tmp, node_scan_tmp}) + 256;
  std::vector<Sl> sl = {
      {(void**)&mv->d_off, sizeof(long long) * (P + 2)}, {(void**)&mv->d_node, sizeof(int32_t) * P * max_ops},
      {(void**)&mv->d_state, P * max_ops}, {(void**)&mv->d_kind, P * max_ops}, {(void**)&mv->d_next, sizeof(int32_t) * P},
      {(void**)&mv->d_key, sizeof(uint32_t) * P}, {(void**)&mv->d_key2, sizeof(uint32_t) * P}, {(void**)&mv->d_val, sizeof(int32_t) * P},
      {(void**)&mv->d_val2, sizeof(int32_t) * P}, {(void**)&mv->d_ncnt, sizeof(int32_t) * (NN + 1)}, {(void**)&mv->d_noff, sizeof(int32_t) * (NN + 2)},
      {(void**)&mv->d_nbest, sizeof(unsigned long long) * NN}, {(void**)&mv->d_best, sizeof(int32_t) * NN}, {(void**)&mv->d_tmp, mv->tmp_bytes},
      {(void**)&d_slot, sizeof(int32_t) * (n_states + 1)}, {(void**)&d_beg, sizeof(int32_t) * P * std::max(SL, 1)},
      {(void**)&d_end, sizeof(int32_t) * P * std::max(SL, 1)}, {(void**)&p_node, sizeof(int32_t) * P * max_ops},
      {(void**)&p_state, P * max_ops}, {(void**)&p_kind, P * max_ops}, {(void**)&d_cnt, sizeof(int32_t) * (P + 1)}};
  size_t total = 0;
  for (auto& x : sl) total += align_up(x.bytes, 256);
  if (cudaMallocAsync((void**)&mv->arena, total, st) != cudaSuccess) { delete mv; return fail(ctx, BLANCE_ERR_NOMEM, "blance_moves_create: device allocation failed"); }
  { size_t off = 0; for (auto& x : sl) { *x.p = mv->arena + off; off += align_up(x.bytes, 256); } }
  int rc = BLANCE_OK;
  auto step = [&](cudaError_t e, const char* what) {
    if (e != cudaSuccess && rc == BLANCE_OK) rc = fail(ctx, BLANCE_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  };
  step(cudaMemcpyAsync(d_slot, state_slot_off, sizeof(int32_t) * (n_states + 1), cudaMemcpyHostToDevice, st), "H2D");
  if (n_parts > 0 && SL > 0) {
    step(cudaMemcpyAsync(d_beg, beg_rows, sizeof(int32_t) * (size_t)n_parts * SL, cudaMemcpyHostToDevice, st), "H2D");
    step(cudaMemcpyAsync(d_end, end_rows, sizeof(int32_t) * (size_t)n_parts * SL, cudaMemcpyHostToDevice, st), "H2D");
  }
  step(cudaMemsetAsync(d_cnt, 0, sizeof(int32_t) * (P + 1), st), "memset");
  if (rc == BLANCE_OK && n_parts > 0) {
    k_calc_moves<<<grid_for(ctx, n_parts, 128), 128, 0, st>>>(n_parts, n_states, n_visit_states, d_slot, d_beg, d_end, favor_min_nodes,
                                                             max_ops, p_node, p_state, p_kind, d_cnt);
    size_t tb = mv->tmp_bytes;
    step(cub::DeviceScan::ExclusiveSum(mv->d_tmp, tb, d_cnt, mv->d_off, n_parts + 1, st), "scan");
    k_moves_compact<<<grid_for(ctx, n_parts, 128), 128, 0, st>>>(n_parts, max_ops, mv->d_off, d_cnt, p_node, p_state, p_kind,
                                                                mv->d_node, mv->d_state, mv->d_kind);
    step(cudaGetLastError(), "k_calc_moves / k_moves_compact");
    ctx->launches += 2;
    step(cudaMemcpyAsync(&mv->total_ops, mv->d_off + n_parts, sizeof(long long), cudaMemcpyDeviceToHost, st), "D2H");
  } else {
    step(cudaMemsetAsync(mv->d_off, 0, sizeof(long long) * (P + 2), st), "memset");
  }
  step(cudaStreamSynchronize(st), "sync");
  if (rc != BLANCE_OK) { cudaFreeAsync(mv->arena, st); delete mv; return rc; }
  if (total_ops) *total_ops = mv->total_ops;
  *out = mv;
  return BLANCE_OK;
}

extern "C" int blance_moves_fetch(blance_ctx* ctx, blance_moves* mv, int64_t* op_off, int32_t* op_node, uint8_t* op_state, uint8_t* op_kind) {
  if (!ctx || !mv) return fail(ctx, BLANCE_ERR_INVALID_ARG, "ctx or moves is NULL");
  if (!ctx->children.empty()) ctx = ctx->children[0];
  std::lock_guard<std::mutex> g(ctx->mu);
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  if (op_off) CK(cudaMemcpyAsync(op_off, mv->d_off, sizeof(long long) * ((size_t)mv->n_parts + 1), cudaMemcpyDeviceToHost, st));
  if (mv->total_ops > 0) {
    if (op_node) CK(cudaMemcpyAsync(op_node, mv->d_node, sizeof(int32_t) * (size_t)mv->total_ops, cudaMemcpyDeviceToHost, st));
    if (op_state) CK(cudaMemcpyAsync(op_state, mv->d_state, (size_t)mv->total_ops, cudaMemcpyDeviceToHost, st));
    if (op_kind) CK(cudaMemcpyAsync(op_kind, mv->d_kind, (size_t)mv->total_ops, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  return BLANCE_OK;
}

extern "C" int blance_moves_available(blance_ctx* ctx, blance_moves* mv, const int32_t* next, int32_t* node_off, int32_t* node_parts,
                                      int32_t* best_part) {
  if (!ctx || !mv || !next) return fail(ctx, BLANCE_ERR_INVALID_ARG, "ctx, moves or next is NULL");
  if (!ctx->children.empty()) ctx = ctx->children[0];
  std::lock_guard<std::mutex> g(ctx->mu);
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int P = mv->n_parts, NN = mv->n_node_ids;
  CK(cudaMemsetAsync(mv->d_ncnt, 0, sizeof(int32_t) * ((size_t)NN + 1), st));
  CK(cudaMemsetAsync(mv->d_nbest, 0xFF, sizeof(unsigned long long) * (size_t)std::max(NN, 1), st));
  if (P > 0) {
    CK(cudaMemcpyAsync(mv->d_next, next, sizeof(int32_t) * (size_t)P, cudaMemcpyHostToDevice, st));
    k_moves_next<<<grid_for(ctx, P, 256), 256, 0, st>>>(P, NN, mv->d_off, mv->d_node, mv->d_kind, mv->d_next, mv->d_key, mv->d_val,
                                                       mv->d_ncnt, mv->d_nbest);
    size_t tb = mv->tmp_bytes;
    CK(cub::DeviceRadixSort::SortPairs(mv->d_tmp, tb, mv->d_key, mv->d_key2, mv->d_val, mv->d_val2, P, 0, 32, st));   // stable: partitions stay ascending
    ctx->launches += 1;
  }
  {
    size_t tb = mv->tmp_bytes;
    CK(cub::DeviceScan::ExclusiveSum(mv->d_tmp, tb, mv->d_ncnt, mv->d_noff, NN + 1, st));
  }
  if (NN > 0) { k_moves_best<<<(NN + 255) / 256, 256, 0, st>>>(NN, mv->d_nbest, mv->d_best); ctx->launches += 1; }
  CK(cudaGetLastError());
  int32_t n_avail = 0;
  CK(cudaMemcpyAsync(&n_avail, mv->d_noff + NN, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (node_off) CK(cudaMemcpyAsync(node_off, mv->d_noff, sizeof(int32_t) * ((size_t)NN + 1), cudaMemcpyDeviceToHost, st));
  if (best_part && NN > 0) CK(cudaMemcpyAsync(best_part, mv->d_best, sizeof(int32_t) * (size_t)NN, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (node_parts && n_avail > 0) {
    CK(cudaMemcpyAsync(node_parts, mv->d_val2, sizeof(int32_t) * (size_t)n_avail, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  return BLANCE_OK;
}

extern "C" void blance_moves_free(blance_ctx* ctx, blance_moves* mv) {
  if (!mv) return;
  if (ctx && !ctx->children.empty()) ctx = ctx->children[0];
  if (ctx) {
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaSetDevice(ctx->device);
    if (mv->arena) cudaFreeAsync(mv->arena, ctx->stream);
    cudaStreamSynchronize(ctx->stream);
  } else if (mv->arena) cudaFree(mv->arena);
  delete mv;
}
